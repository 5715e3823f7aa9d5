// C ABI of the batched simulator (include/pgw.h): owns the device-side tables and
// state of one env batch and sequences the kernels of reset / step.
//
//   reset:  [power flow, base load only]  ->  [component reset kernel]
//   step:   [component step kernel]       ->  [power flow + reward hook]
//
// The episode clock lives on the device and is advanced by the last CTA of the last
// kernel of a step, so a step has constant launch parameters (CUDA-graph friendly).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <new>
#include <string>
#include <vector>

#include "internal.cuh"
#include "tables.h"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define PGW_CUDA(expr)                                                                  \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess)                                                              \
      return fail(PGW_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));   \
  } while (0)

template <typename T>
cudaError_t upload(T** dst, const T* src, size_t n) {
  *dst = nullptr;
  if (n == 0) return cudaSuccess;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(dst), n * sizeof(T));
  if (e != cudaSuccess) return e;
  return cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice);
}

template <typename T>
cudaError_t alloc_zero(T** dst, size_t n) {
  *dst = nullptr;
  if (n == 0) return cudaSuccess;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(dst), n * sizeof(T));
  if (e != cudaSuccess) return e;
  return cudaMemset(*dst, 0, n * sizeof(T));
}

}  // namespace

struct pgw_env {
  int E = 0, A = 0, C = 0, act_dim = 0, obs_dim = 0, sd_rows = 0, si_rows = 0;
  int num_storage = 0, num_events = 0, dpar_len = 0;
  bool has_feeder = false;
  bool need_scratch = false, need_scratch_reset = false;
  int pf_kernel = 0;
  int clock = -1;             // host mirror
  long long resets = 0;
  long long launches = 0;
  long long graph_captures = 0;        // graphs captured + instantiated since creation
  // Launch parameters of the whole batch (tables built by tables.cpp, device pointers of this
  // handle): every launch copies its kernel's base and sets the fields of the call
  pgw::CompParams comp_base{};
  pgw::PfParams pf_base{};
  bool warm_start = true;
  bool tc2_tol_set = false;             // PGW_OPT_PF_TC_TOL_NANO was given: the polish option leaves tol alone
  pgw::Tc2Consts tc2c{};                // pf_base.tc2.consts / pconsts point here
  pgw::Tc2Polish tc2p{};
  // device tables
  unsigned char* comp_blob = nullptr;   // [agents | comps | dpar | ipar]
  double* dtab = nullptr;
  int32_t* itab = nullptr;
  // The captured CUDA graph of a step: ONE per handle and I/O form (float64 / float32 actions and
  // observations, [io32]); its kernel nodes are re-pointed at the caller's buffers when those change
  // (kind: 0 fused step, 1 components, 2 power flow)
  struct StepGraph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    cudaGraphNode_t nodes[2] = {nullptr, nullptr};
    cudaKernelNodeParams params[2] = {};
    int kind[2] = {0, 0}, nargs[2] = {1, 1}, num_nodes = 0, pdl = 0;
    bool has_event = false;             // the fused node's parameters carry a host-side event index
    const void *actions = nullptr, *obs = nullptr, *rew = nullptr, *done = nullptr;
    void destroy() {
      if (exec) cudaGraphExecDestroy(exec);
      if (graph) cudaGraphDestroy(graph);
      exec = nullptr; graph = nullptr; num_nodes = 0;
    }
  };
  StepGraph step_graph[2];
  // graphs of the pipelined host-buffer step, keyed by the host pointers (memcpy nodes) and I/O form
  struct HostGraph {
    const void *actions, *obs, *rew, *done;
    bool io32;
    cudaGraphExec_t exec;
  };
  std::vector<HostGraph> host_graphs;
  static constexpr int kMaxChunks = 8;
  int host_chunks = 0;                  // PGW_OPT_HOST_CHUNKS: 0 = automatic
  bool host_zero_copy = true;           // PGW_OPT_HOST_ZERO_COPY
  // device views of the caller's host buffers (cudaPointerGetAttributes is a driver query:
  // remembered per pointer; nullptr = not page-locked / not device accessible)
  struct HostView { const void* host; void* dev; };
  std::vector<HostView> host_views;
  cudaStream_t chunk_stream[kMaxChunks] = {};
  cudaEvent_t ev_fork = nullptr, ev_join[kMaxChunks] = {};
  void drop_graphs() {
    step_graph[0].destroy();
    step_graph[1].destroy();
    for (auto& g : host_graphs) cudaGraphExecDestroy(g.exec);
    host_graphs.clear();
  }
  bool use_graphs = true;
  bool use_pdl = true;
  // fused step kernel (step_fused.cu): eligible scenario, and PGW_OPT_FUSED (0 off, 1 auto: batches
  // of at most two 32-env tiles per SM, 2 always)
  bool fused_ok = false;
  int fused_mode = 1;
  bool clip_init_soc = true;
  // device state
  double* sd = nullptr;
  double2* u_state = nullptr;           // [nbp][E] power-flow warm start
  uint32_t* si = nullptr;
  double *agent_p = nullptr, *ep_ret = nullptr, *rew_last = nullptr;
  double *vmag = nullptr, *vmin = nullptr, *vmax = nullptr, *vbus = nullptr, *viol = nullptr;
  int32_t* iters = nullptr;
  int* d_clock = nullptr;
  unsigned int* d_ticket = nullptr;
  long long* phase_clk = nullptr;       // PGW_PHASE_TIMERS builds (tools/phase_probe.py)
  // staging for the *_host entry points
  double *h_act = nullptr, *h_obs = nullptr, *h_rew = nullptr, *h_soc = nullptr;
  float *h_act32 = nullptr, *h_obs32 = nullptr;   // float32 I/O (the *_f32 entry points)
  uint8_t* h_done = nullptr;
  std::vector<void*> owned;
  // optional per-kernel timing (pgw_set_timing)
  bool timing = false;
  std::vector<cudaEvent_t> ev_pool;     // triples: start, after components, after power flow
  size_t ev_used = 0;
  double t_comp_ms = 0, t_pf_ms = 0, t_steps = 0;

  ~pgw_env() {
    for (void* p : owned) cudaFree(p);
    for (cudaEvent_t e : ev_pool) cudaEventDestroy(e);
    drop_graphs();
    if (ev_fork) cudaEventDestroy(ev_fork);
    for (int k = 0; k < kMaxChunks; ++k) {
      if (ev_join[k]) cudaEventDestroy(ev_join[k]);
      if (chunk_stream[k]) cudaStreamDestroy(chunk_stream[k]);
    }
  }
  cudaEvent_t next_event() {
    if (ev_used == ev_pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      ev_pool.push_back(e);
    }
    return ev_pool[ev_used++];
  }
  template <typename T>
  void own(T* p) {
    if (p) owned.push_back(const_cast<void*>(reinterpret_cast<const void*>(p)));
  }
};

extern "C" {

const char* pgw_last_error(void) { return g_err.c_str(); }
int pgw_abi_version(void) { return PGW_ABI_VERSION; }

int pgw_create(const pgw_spec* spec, pgw_env** out) {
  if (!spec || !out) return fail(PGW_ERR_INVALID, "null argument");
  *out = nullptr;
  if (const std::string bad = pgw::validate_spec(*spec); !bad.empty()) return fail(PGW_ERR_INVALID, bad);
  // 16 CTAs per SM (10 are resident: 96 registers x 64 threads) lets the hardware scheduler
  // even out the rough cost estimates of a many-agent scenario (C3: 134 us at 16 per SM,
  // 150 us at 10); with a single agent there is nothing to even out and a second round of
  // CTAs only adds a partial wave (262 144 houses: 42.3 us at 16 per SM, 35.8 us at 10).
  int budget = spec->num_agents == 1 ? 148 * 10 : 148 * 16;
  if (const char* b = getenv("PGW_CTA_BUDGET")) budget = std::max(1, atoi(b));   // tuning knob
  pgw::CompTables ct = pgw::build_comp_tables(*spec, budget);
  if (pgw::comp_staging_bytes(ct.base) > 160 * 1024)
    return fail(PGW_ERR_INVALID, "scenario tables exceed the shared-memory staging budget");
  pgw::FeederTables ft;
  if (spec->feeder) {
    ft = pgw::build_feeder_tables(*spec, pgw::tc2_padded_chunks((spec->feeder->nb + 7) / 8));
    if (!ft.error.empty()) return fail(PGW_ERR_INVALID, ft.error);
  }
  int dev = 0;
  PGW_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  PGW_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(PGW_ERR_ARCH, "this library is built for sm_100a (B200) only");

  pgw_env* env = new (std::nothrow) pgw_env();
  if (!env) return fail(PGW_ERR_NOMEM, "host allocation failed");
  env->E = spec->num_envs; env->A = spec->num_agents; env->C = spec->num_components;
  env->act_dim = spec->act_dim; env->obs_dim = spec->obs_dim;
  env->sd_rows = spec->sd_rows; env->si_rows = spec->si_rows;
  env->num_storage = spec->num_storage; env->num_events = spec->num_events; env->dpar_len = spec->dpar_len;
  env->need_scratch = ct.need_scratch; env->need_scratch_reset = ct.need_scratch_reset;
  const size_t E = (size_t)env->E, A = (size_t)env->A;

#define PGW_TRY(expr)                                                                  \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      delete env;                                                                      \
      return fail(_e == cudaErrorMemoryAllocation ? PGW_ERR_NOMEM : PGW_ERR_CUDA,      \
                  std::string(#expr) + ": " + cudaGetErrorString(_e));                 \
    }                                                                                  \
  } while (0)

  pgw::CtaWork* work = nullptr;
  PGW_TRY(upload(&env->comp_blob, ct.blob.data(), ct.blob.size())); env->own(env->comp_blob);
  PGW_TRY(upload(&work, ct.work.data(), ct.work.size())); env->own(work);
  PGW_TRY(upload(&env->dtab, spec->dtab, (size_t)spec->num_events * spec->dtab_stride)); env->own(env->dtab);
  PGW_TRY(upload(&env->itab, spec->itab, (size_t)spec->num_events * spec->itab_stride)); env->own(env->itab);

  PGW_TRY(alloc_zero(&env->sd, (size_t)env->sd_rows * E)); env->own(env->sd);
  PGW_TRY(alloc_zero(&env->si, (size_t)env->si_rows * E)); env->own(env->si);
  PGW_TRY(alloc_zero(&env->agent_p, A * E)); env->own(env->agent_p);
  PGW_TRY(alloc_zero(&env->ep_ret, A * E)); env->own(env->ep_ret);
  PGW_TRY(alloc_zero(&env->rew_last, A * E)); env->own(env->rew_last);
  PGW_TRY(alloc_zero(&env->d_clock, 1)); env->own(env->d_clock);
  PGW_TRY(alloc_zero(&env->d_ticket, 1)); env->own(env->d_ticket);
#ifdef PGW_PHASE_TIMERS
  PGW_TRY(alloc_zero(&env->phase_clk, (size_t)4096 * 16 + (size_t)4096 * 8)); env->own(env->phase_clk);
#endif

  pgw::PfParams& pf = env->pf_base;
  if (spec->feeder) {
    env->has_feeder = true;
    pf = ft.base; env->tc2c = ft.tc2c; env->tc2p = ft.tc2p;
    unsigned char* blob = nullptr;
    PGW_TRY(upload(&blob, ft.blob.data(), ft.blob.size())); env->own(pf.blob = blob);
    PGW_TRY(alloc_zero(&env->u_state, (size_t)pf.nbp * E)); env->own(env->u_state);
    PGW_TRY(upload(&blob, ft.tc_blob.data(), ft.tc_blob.size())); env->own(pf.tc_blob = blob);
    if (!ft.tc2_blob.empty()) {
      // the handle's own copies, passed to the tc2 kernel as __grid_constant__ parameters
      pf.tc2.consts = &env->tc2c;
      if (pf.tc2.polish_ok) pf.tc2.pconsts = &env->tc2p;
      if (pgw::tc2_smem_bytes(pf) + 6 * 1024 <= 227 * 1024) {   // + the kernel's static arrays
        PGW_TRY(upload(&blob, ft.tc2_blob.data(), ft.tc2_blob.size())); env->own(pf.tc2.blob = blob);
        // The fused step kernel serves feeders with <= 16 load branches, stock components on their
        // straight-line paths, tables that fit shared memory.
        bool ok = pf.tc2.nch == 2 && !ct.base.has_house && !ct.base.ev_per_env && !env->need_scratch;
        for (int c = 0; c < spec->num_components && ok; ++c) {
          const pgw_component& k = spec->components[c];
          ok = k.type >= PGW_STORAGE && k.type <= PGW_BUILDING &&
               (k.type != PGW_BUILDING || (k.flags & PGW_F_BUILDING_FAST));
        }
        if (ok) {
          pgw::FusedParams P{};
          P.c = ct.base; P.f = pf; P.C = env->C; P.act_dim = env->act_dim;
          ok = pgw::step_fused_smem_bytes(P) + 2048 <= 200 * 1024;
        }
        env->fused_ok = ok;
      }
    }
    PGW_TRY(alloc_zero(&env->vmag, (size_t)pf.nn * E)); env->own(env->vmag);
    PGW_TRY(alloc_zero(&env->vmin, E)); env->own(env->vmin);
    PGW_TRY(alloc_zero(&env->vmax, E)); env->own(env->vmax);
    PGW_TRY(alloc_zero(&env->vbus, A * E)); env->own(env->vbus);
    PGW_TRY(alloc_zero(&env->viol, E)); env->own(env->viol);
    PGW_TRY(alloc_zero(&env->iters, E)); env->own(env->iters);
  }
#undef PGW_TRY
  pgw::CompParams& cp = env->comp_base = ct.base;
  cp.blob = env->comp_blob; cp.work = work; cp.dtab = env->dtab; cp.itab = env->itab; cp.sd = env->sd; cp.si = env->si;
  cp.rew_copy = env->rew_last; cp.vmin = env->vmin; cp.vmax = env->vmax; cp.vbus = env->vbus;
  cp.agent_p = env->agent_p; cp.ep_ret = env->ep_ret; cp.clock = env->d_clock; cp.ticket = env->d_ticket;
  pf.u_state = env->u_state; pf.rew_copy = env->rew_last; pf.dtab = env->dtab; pf.vmag = env->vmag;
  pf.vmin = env->vmin; pf.vmax = env->vmax; pf.vbus = env->vbus; pf.iters = env->iters; pf.ep_ret = env->ep_ret;
  pf.viol = env->viol; pf.clock = env->d_clock; pf.ticket = env->d_ticket;
#ifdef PGW_PHASE_TIMERS
  cp.phase_clk = env->phase_clk + (size_t)4096 * 16;
  pf.phase_clk = env->phase_clk;
#endif
  *out = env;
  return PGW_OK;
}

int pgw_destroy(pgw_env* env) {
  if (!env) return PGW_OK;
  if (env->h_act) cudaFree(env->h_act);
  if (env->h_obs) cudaFree(env->h_obs);
  if (env->h_act32) cudaFree(env->h_act32);
  if (env->h_obs32) cudaFree(env->h_obs32);
  if (env->h_rew) cudaFree(env->h_rew);
  if (env->h_soc) cudaFree(env->h_soc);
  if (env->h_done) cudaFree(env->h_done);
  delete env;
  return PGW_OK;
}

static int pf_grid(const pgw_env* env, const pgw::PfParams& pf) {
  if (env->pf_kernel == 2) return pgw::tc2_grid(pf);
  return env->pf_kernel == 1 ? pgw::tc_grid(pf) : pgw::fp64_grid(pf);
}

// pf.tickets == 0: this launch is the only one of its kind in the step
static cudaError_t launch_pf(const pgw_env* env, pgw::PfParams pf, cudaStream_t s) {
  if (pf.tickets == 0u) pf.tickets = (unsigned int)pf_grid(env, pf);
  if (env->pf_kernel == 2) return pgw::launch_powerflow_tc2(pf, s);
  return env->pf_kernel == 1 ? pgw::launch_powerflow_tc(pf, s) : pgw::launch_powerflow(pf, s);
}

static int smem_for_events(const pgw_env* env, bool reset = false) {
  // static blob | event rows | per-thread scratch (component_math.cuh kScratchDoubles x 64
  // threads; only the table-driven building path uses it)
  return pgw::comp_staging_bytes(env->comp_base) +
         ((reset ? env->need_scratch_reset : env->need_scratch) ? 35 * 64 * 8 : 0);
}

// io32: obs is a float array (pgw_reset_f32), else double
static int reset_impl(pgw_env* env, const double* init_soc, void* obs, bool io32, void* cuda_stream) {
  if (!env || !obs) return fail(PGW_ERR_INVALID, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  PGW_CUDA(cudaMemsetAsync(env->d_clock, 0, sizeof(int), s));
  PGW_CUDA(cudaMemsetAsync(env->d_ticket, 0, sizeof(unsigned int), s));
  if (env->has_feeder) {
    pgw::PfParams pf = env->pf_base;
    pf.event_mode = 0; pf.advance_clock = 0; pf.agent_p = nullptr; pf.rew = nullptr;
    pf.punit = 0.0; pf.warm_start = 0;
    PGW_CUDA(launch_pf(env, pf, s));
    ++env->launches;
  }
  pgw::CompParams cp = env->comp_base;
  cp.event_mode = 0; cp.advance_clock = 0; cp.init_soc = init_soc; cp.obs = obs; cp.io32 = io32 ? 1 : 0;
  cp.clip_init_soc = env->clip_init_soc ? 1 : 0;
  cp.first_reset = env->resets == 0 ? 1 : 0;
  ++env->resets;
  PGW_CUDA(pgw::launch_components(cp, smem_for_events(env, true), s));
  ++env->launches;
  env->clock = 0;
  return PGW_OK;
}

int pgw_reset(pgw_env* env, const double* init_soc, double* obs, void* cuda_stream) {
  return reset_impl(env, init_soc, obs, false, cuda_stream);
}

int pgw_reset_f32(pgw_env* env, const double* init_soc, float* obs, void* cuda_stream) {
  return reset_impl(env, init_soc, obs, true, cuda_stream);
}

// ---- launch parameters of the kernels of one step over the envs [e_lo, e_hi)
static pgw::CompParams step_comp_params(pgw_env* env, const void* actions, void* obs, double* rew,
                                        uint8_t* done, bool io32, int e_lo, int e_hi, int chunks,
                                        int pdl_trigger) {
  pgw::CompParams cp = env->comp_base;
  const bool hook = env->has_feeder && env->pf_base.punit != 0.0;   // power flow finishes the rewards
  cp.event_mode = 1; cp.advance_clock = env->has_feeder ? 0 : 1; cp.owns_reward = hook ? 0 : 1;
  cp.actions = actions; cp.obs = obs; cp.rew = rew; cp.done = done; cp.io32 = io32 ? 1 : 0;
  cp.pdl_trigger = pdl_trigger;
  cp.e_lo = e_lo; cp.e_hi = e_hi; cp.tickets = (unsigned int)(cp.num_ctas * chunks);
  return cp;
}

// Programmatic dependent launch of the tcgen05 power-flow kernel behind the component kernel.
// Used when a power-flow CTA leaves room on its SM (IEEE-13 class feeders); a CTA that fills the
// SM's shared memory gains nothing from starting early and was measured 2 us slower per step at
// C3.  The component kernel releases the dependent right after its clock read when both grids fit
// on the GPU side by side (1), else at the end of each CTA (2).
// Measured (C1, cold L2): 27.5 -> 25.6 us per step at 4096 envs, 40.1 -> 37.9 us at 32 768.
static int pdl_trigger_mode(const pgw_env* env, bool timed) {
  if (!env->use_pdl || timed || !env->has_feeder || env->pf_kernel != 2) return 0;
  pgw::PfParams pf = env->pf_base;
  pf.event_mode = 1; pf.reward_hook = (pf.punit != 0.0) ? 1 : 0;
  if (pgw::tc2_smem_bytes(pf) > 112 * 1024) return 0;   // two power-flow CTAs + component CTAs per SM
  return env->comp_base.num_ctas <= 148 * 4 ? 1 : 2;
}

static pgw::PfParams step_pf_params(pgw_env* env, double* rew, int e_lo, int e_hi, unsigned int tickets,
                                    bool pdl) {
  pgw::PfParams pf = env->pf_base;
  pf.event_mode = 1; pf.advance_clock = 1; pf.agent_p = env->agent_p; pf.rew = rew;
  pf.reward_hook = (pf.punit != 0.0) ? 1 : 0;
  pf.pdl = pdl ? 1 : 0;
  pf.warm_start = env->warm_start ? 1 : 0;
  pf.e_lo = e_lo; pf.e_hi = e_hi;
  pf.tickets = tickets ? tickets : (unsigned int)pf_grid(env, pf);
  return pf;
}

static bool use_fused(const pgw_env* env) {
  if (!env->fused_ok || env->pf_kernel != 2 || env->fused_mode == 0) return false;
  return env->fused_mode == 2 || pgw::step_fused_tiles(env->E) <= 2 * 148;
}

static int fused_grid(int envs) {
  static const int cap = [] {                          // PGW_FUSED_GRID: tuning knob (CTAs of the fused kernel)
    const char* v = getenv("PGW_FUSED_GRID");
    return v ? std::max(1, atoi(v)) : 148;
  }();
  return std::max(1, std::min(pgw::step_fused_tiles(envs), cap));
}

// `tickets` = CTAs of all the launches that make up the step (the CTA that takes the last ticket
// advances the clock); 0 = this launch is the whole step.
static pgw::FusedParams step_fused_params(pgw_env* env, const void* actions, void* obs, double* rew,
                                          uint8_t* done, bool io32, int e_lo, int e_hi, unsigned int tickets,
                                          int stagger = 0, int event = -1) {
  pgw::FusedParams P{};
  P.event = event;
  P.c = step_comp_params(env, actions, obs, rew, done, io32, e_lo, e_hi, 1, 0);
  P.f = step_pf_params(env, rew, e_lo, e_hi, 1u, false);
  P.C = env->C; P.act_dim = env->act_dim; P.sd_rows = env->sd_rows; P.e_lo = e_lo; P.e_hi = e_hi;
  P.tickets = tickets ? tickets : (unsigned int)fused_grid(e_hi - e_lo);
  P.stagger_cycles = stagger;
  return P;
}

// The kernels of one step over [e_lo, e_hi), enqueued on `s` (directly, or while `s` is being
// captured).  chunks = launches of this kind that make up the step (pgw_step_host pipelines
// env chunks); their CTA counts add up to the clock tickets.
static unsigned int step_pf_tickets(pgw_env* env, const int* bounds, int chunks) {
  unsigned int n = 0;
  for (int k = 0; k < chunks; ++k) {
    if (use_fused(env)) {
      n += (unsigned int)fused_grid(bounds[k + 1] - bounds[k]);
    } else {
      pgw::PfParams pf = env->pf_base;
      pf.event_mode = 1; pf.reward_hook = (pf.punit != 0.0) ? 1 : 0;
      pf.e_lo = bounds[k]; pf.e_hi = bounds[k + 1];
      n += (unsigned int)pf_grid(env, pf);
    }
  }
  return n;
}

static int enqueue_step(pgw_env* env, const void* actions, void* obs, double* rew,
                        uint8_t* done, bool io32, cudaStream_t s, bool timed, int e_lo = 0, int e_hi = -1,
                        int chunks = 1, unsigned int pf_tickets = 0u, int stagger = 0, int event = -1) {
  if (e_hi < 0) e_hi = env->E;
  if (use_fused(env)) {
    if (timed) PGW_CUDA(cudaEventRecord(env->next_event(), s));
    const pgw::FusedParams P = step_fused_params(env, actions, obs, rew, done, io32, e_lo, e_hi, pf_tickets, stagger,
                                                 event);
    PGW_CUDA(pgw::launch_step_fused(P, fused_grid(e_hi - e_lo), s));
    if (timed) {                                       // one kernel: reported in the component slot
      PGW_CUDA(cudaEventRecord(env->next_event(), s));
      PGW_CUDA(cudaEventRecord(env->next_event(), s));
    }
    return PGW_OK;
  }
  const int pdl = chunks == 1 ? pdl_trigger_mode(env, timed) : 0;
  if (timed) PGW_CUDA(cudaEventRecord(env->next_event(), s));
  PGW_CUDA(pgw::launch_components(step_comp_params(env, actions, obs, rew, done, io32, e_lo, e_hi, chunks, pdl),
                                  smem_for_events(env), s));
  if (timed) PGW_CUDA(cudaEventRecord(env->next_event(), s));
  if (env->has_feeder)
    PGW_CUDA(launch_pf(env, step_pf_params(env, rew, e_lo, e_hi, pf_tickets, pdl != 0), s));
  if (timed) PGW_CUDA(cudaEventRecord(env->next_event(), s));
  return PGW_OK;
}

static int step_kernels(const pgw_env* env) { return use_fused(env) ? 1 : (env->has_feeder ? 2 : 1); }

// Re-point the kernel nodes of the captured step graph at another set of caller buffers
// (cudaGraphExecKernelNodeSetParams: no re-capture, no re-instantiation; a policy loop that
// hands in a fresh action tensor every step replays the same executable graph).
static int retarget_step_graph(pgw_env* env, const void* actions, void* obs, double* rew,
                               uint8_t* done, bool io32, int event) {
  pgw_env::StepGraph& g = env->step_graph[io32];
  for (int i = 0; i < g.num_nodes; ++i) {
    cudaKernelNodeParams np = g.params[i];
    void* args[4] = {nullptr, nullptr, nullptr, nullptr};
    for (int q = 1; q < g.nargs[i]; ++q) args[q] = g.params[i].kernelParams[q];
    pgw::FusedParams fp;
    pgw::CompParams cp;
    pgw::PfParams pf;
    if (g.kind[i] == 0) {
      fp = step_fused_params(env, actions, obs, rew, done, io32, 0, env->E, 0u, 0, event);
      args[0] = &fp;
      g.has_event = event >= 0;
    } else if (g.kind[i] == 1) {
      cp = step_comp_params(env, actions, obs, rew, done, io32, 0, env->E, 1, g.pdl);
      args[0] = &cp;
    } else {
      pf = step_pf_params(env, rew, 0, env->E, 0u, g.pdl != 0);
      args[0] = &pf;
    }
    np.kernelParams = args;
    np.extra = nullptr;
    PGW_CUDA(cudaGraphExecKernelNodeSetParams(g.exec, g.nodes[i], &np));
  }
  g.actions = actions; g.obs = obs; g.rew = rew; g.done = done;
  return PGW_OK;
}

static int capture_step_graph(pgw_env* env, const void* actions, void* obs, double* rew,
                              uint8_t* done, bool io32, cudaStream_t s) {
  pgw_env::StepGraph& g = env->step_graph[io32];
  g.destroy();
  g.pdl = pdl_trigger_mode(env, false);
  PGW_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  int rc = enqueue_step(env, actions, obs, rew, done, io32, s, false);
  cudaError_t ce = cudaStreamEndCapture(s, &g.graph);
  if (rc != PGW_OK) { g.destroy(); return rc; }
  if (ce != cudaSuccess) {
    g.destroy();
    return fail(PGW_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce));
  }
  ce = cudaGraphInstantiate(&g.exec, g.graph, 0);
  if (ce != cudaSuccess) {
    g.destroy();
    return fail(PGW_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce));
  }
  cudaGraphNode_t nodes[8];
  size_t n = 8;
  PGW_CUDA(cudaGraphGetNodes(g.graph, nodes, &n));
  g.num_nodes = 0;
  for (size_t i = 0; i < n; ++i) {
    cudaGraphNodeType ty;
    PGW_CUDA(cudaGraphNodeGetType(nodes[i], &ty));
    if (ty != cudaGraphNodeTypeKernel) continue;
    if (g.num_nodes == 2) { g.destroy(); return fail(PGW_ERR_CUDA, "unexpected step graph"); }
    const int q = g.num_nodes++;
    g.nodes[q] = nodes[i];
    PGW_CUDA(cudaGraphKernelNodeGetParams(nodes[i], &g.params[q]));
    if (pgw::is_step_fused_kernel(g.params[q].func)) { g.kind[q] = 0; g.nargs[q] = 1; }
    else if (pgw::is_component_kernel(g.params[q].func)) { g.kind[q] = 1; g.nargs[q] = 1; }
    else { g.kind[q] = 2; g.nargs[q] = env->pf_kernel == 2 ? 3 : 1; }
  }
  g.actions = actions; g.obs = obs; g.rew = rew; g.done = done;
  g.has_event = false;
  ++env->graph_captures;
  return PGW_OK;
}

static int step_impl(pgw_env* env, const void* actions, void* obs, double* rew, uint8_t* done, bool io32,
                     void* cuda_stream) {
  if (!env || !actions || !obs || !rew || !done) return fail(PGW_ERR_INVALID, "null argument");
  if (env->clock < 0) return fail(PGW_ERR_STATE, "pgw_step before pgw_reset");
  if (env->clock + 1 >= env->num_events)
    return fail(PGW_ERR_STATE, "episode is over: call pgw_reset");
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);

  // Replay the captured graph of the step (the episode clock lives on the device, so the launch
  // parameters of a step change only with the caller's buffers, and those are patched in place).
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  PGW_CUDA(cudaStreamIsCapturing(s, &cap));
  const bool graphable = env->use_graphs && !env->timing && cap == cudaStreamCaptureStatusNone &&
                         s != nullptr;
  if (graphable) {
    pgw_env::StepGraph& g = env->step_graph[io32];
    int rc = PGW_OK;
    if (!g.exec) rc = capture_step_graph(env, actions, obs, rew, done, io32, s);
    else if (g.actions != actions || g.obs != obs || g.rew != rew || g.done != done)
      // the node parameters are rewritten anyway: the step's event index rides along and the
      // fused kernel skips its read of the device clock
      rc = retarget_step_graph(env, actions, obs, rew, done, io32, env->clock + 1);
    else if (g.has_event)                              // same buffers again: back to the device clock
      rc = retarget_step_graph(env, actions, obs, rew, done, io32, -1);
    if (rc != PGW_OK) return rc;
    PGW_CUDA(cudaGraphLaunch(g.exec, s));
  } else {
    // direct launches know the event index; a launch recorded into the CALLER's capture is
    // replayed with frozen parameters and has to read the device clock
    const int event = cap == cudaStreamCaptureStatusNone ? env->clock + 1 : -1;
    int rc = enqueue_step(env, actions, obs, rew, done, io32, s, env->timing, 0, -1, 1, 0u, 0, event);
    if (rc != PGW_OK) return rc;
  }
  env->launches += step_kernels(env);
  ++env->clock;
  return PGW_OK;
}

int pgw_step(pgw_env* env, const double* actions, double* obs, double* rew, uint8_t* done,
             void* cuda_stream) {
  return step_impl(env, actions, obs, rew, done, false, cuda_stream);
}

int pgw_step_f32(pgw_env* env, const float* actions, float* obs, double* rew, uint8_t* done,
                 void* cuda_stream) {
  return step_impl(env, actions, obs, rew, done, true, cuda_stream);
}

// device staging of the host-buffer entry points: actions / observations in the I/O form's element type
static int ensure_staging(pgw_env* env, bool io32) {
  const size_t E = (size_t)env->E;
  if (io32) {
    if (!env->h_act32) PGW_CUDA(cudaMalloc(&env->h_act32, (size_t)env->act_dim * E * 4));
    if (!env->h_obs32) PGW_CUDA(cudaMalloc(&env->h_obs32, (size_t)env->obs_dim * E * 4));
  } else {
    if (!env->h_act) PGW_CUDA(cudaMalloc(&env->h_act, (size_t)env->act_dim * E * 8));
    if (!env->h_obs) PGW_CUDA(cudaMalloc(&env->h_obs, (size_t)env->obs_dim * E * 8));
  }
  if (!env->h_rew) PGW_CUDA(cudaMalloc(&env->h_rew, (size_t)env->A * E * 8));
  if (!env->h_done) PGW_CUDA(cudaMalloc(&env->h_done, E));
  if (!env->h_soc && env->num_storage)
    PGW_CUDA(cudaMalloc(&env->h_soc, (size_t)env->num_storage * E * 8));
  return PGW_OK;
}

static int reset_host_impl(pgw_env* env, const double* init_soc, void* obs, bool io32, void* cuda_stream) {
  if (!env || !obs) return fail(PGW_ERR_INVALID, "null argument");
  int rc = ensure_staging(env, io32);
  if (rc) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  const size_t E = (size_t)env->E;
  if (init_soc && env->num_storage)
    PGW_CUDA(cudaMemcpyAsync(env->h_soc, init_soc, (size_t)env->num_storage * E * 8,
                             cudaMemcpyHostToDevice, s));
  void* stage = io32 ? (void*)env->h_obs32 : (void*)env->h_obs;
  rc = reset_impl(env, (init_soc && env->num_storage) ? env->h_soc : nullptr, stage, io32, s);
  if (rc) return rc;
  PGW_CUDA(cudaMemcpyAsync(obs, stage, (size_t)env->obs_dim * E * (io32 ? 4 : 8), cudaMemcpyDeviceToHost, s));
  PGW_CUDA(cudaStreamSynchronize(s));
  return PGW_OK;
}

int pgw_reset_host(pgw_env* env, const double* init_soc, double* obs, void* cuda_stream) {
  return reset_host_impl(env, init_soc, obs, false, cuda_stream);
}

int pgw_reset_host_f32(pgw_env* env, const double* init_soc, float* obs, void* cuda_stream) {
  return reset_host_impl(env, init_soc, obs, true, cuda_stream);
}

// ---- end-to-end step with host buffers, pipelined over env chunks.
// Chunk k: actions of its envs in (a strided copy over the rows x E pitch), the step's kernels on
// that env range, observations / rewards / done flags out -- every chunk on a stream of its own,
// so that the copy-in of chunk k+1, the kernels of chunk k and the copy-out of chunk k-1 overlap
// (PCIe is full duplex, the copy engines are independent of the SMs).  The whole fork-join is
// captured once per set of host buffers and replayed as one graph launch.
static int host_chunks(const pgw_env* env, bool io32) {
  if (env->timing || (env->has_feeder && env->pf_kernel == 1)) return 1;   // kernel 1 has no env ranges
  if (env->host_chunks > 0) return std::min(env->host_chunks, pgw_env::kMaxChunks);
  // Every copy costs ~8 us of fixed latency on top of its bytes (measured, C1: 94 us per step
  // with one chunk, 120 with four): chunks pay off only when a chunk's copy-out is several MB
  const size_t out = (size_t)env->obs_dim * (size_t)env->E * (io32 ? 4 : 8);
  return out >= ((size_t)32 << 20) ? 4 : 1;
}

// Device-side address of a host buffer if the GPU can access it in place (page-locked memory
// under unified addressing: cudaHostAlloc / cudaHostRegister, e.g. torch pin_memory()), else null.
static void* device_view(pgw_env* env, const void* host) {
  for (const auto& v : env->host_views)
    if (v.host == host) return v.dev;
  void* dev = nullptr;
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost)
    dev = at.devicePointer;
  else
    cudaGetLastError();                                // pageable memory: not an error of ours
  if (env->host_views.size() < 64) env->host_views.push_back({host, dev});
  return dev;
}

static int enqueue_host_step(pgw_env* env, const void* actions, void* obs, double* rew,
                             uint8_t* done, bool io32, cudaStream_t s) {
  const int E = env->E;
  int nch = host_chunks(env, io32);
  int bounds[pgw_env::kMaxChunks + 1];
  const int per = ((E + nch - 1) / nch + 127) / 128 * 128;          // whole 128-env tiles
  // Whole tiles can leave the last chunks empty (600 envs in 4 chunks: 256 + 256 + 88 + 0).  An
  // empty chunk launches nothing, so it must not count towards the clock tickets either.
  nch = (E + per - 1) / per;
  for (int k = 0; k <= nch; ++k) bounds[k] = std::min(E, k * per);
  const unsigned int tickets = env->has_feeder ? step_pf_tickets(env, bounds, nch) : 0u;
  const size_t pitch = (size_t)E * 8, esz = io32 ? 4 : 8, io_pitch = (size_t)E * esz;
  unsigned char* act_stage = io32 ? (unsigned char*)env->h_act32 : (unsigned char*)env->h_act;
  unsigned char* obs_stage = io32 ? (unsigned char*)env->h_obs32 : (unsigned char*)env->h_obs;
  if (nch > 1) PGW_CUDA(cudaEventRecord(env->ev_fork, s));
  for (int k = 0; k < nch; ++k) {
    const int e0 = bounds[k], e1 = bounds[k + 1];
    if (e1 <= e0) continue;
    cudaStream_t ck = nch > 1 ? env->chunk_stream[k] : s;
    if (nch > 1) PGW_CUDA(cudaStreamWaitEvent(ck, env->ev_fork, 0));
    const size_t w8 = (size_t)(e1 - e0) * 8, wio = (size_t)(e1 - e0) * esz, o0 = (size_t)e0 * esz;
    PGW_CUDA(cudaMemcpy2DAsync(act_stage + o0, io_pitch, static_cast<const unsigned char*>(actions) + o0, io_pitch,
                               wio, (size_t)env->act_dim, cudaMemcpyHostToDevice, ck));
    int rc = enqueue_step(env, act_stage, obs_stage, env->h_rew, env->h_done, io32, ck, env->timing, e0, e1,
                          nch, tickets);
    if (rc) return rc;
    PGW_CUDA(cudaMemcpy2DAsync(static_cast<unsigned char*>(obs) + o0, io_pitch, obs_stage + o0, io_pitch, wio,
                               (size_t)env->obs_dim, cudaMemcpyDeviceToHost, ck));
    PGW_CUDA(cudaMemcpy2DAsync(rew + e0, pitch, env->h_rew + e0, pitch, w8, (size_t)env->A,
                               cudaMemcpyDeviceToHost, ck));
    PGW_CUDA(cudaMemcpyAsync(done + e0, env->h_done + e0, (size_t)(e1 - e0), cudaMemcpyDeviceToHost, ck));
    if (nch > 1) {
      PGW_CUDA(cudaEventRecord(env->ev_join[k], ck));
      PGW_CUDA(cudaStreamWaitEvent(s, env->ev_join[k], 0));
    }
  }
  return PGW_OK;
}

// The step on page-locked host buffers the GPU addresses in place.  With the fused kernel the
// batch runs as a chain of env chunks on one stream, each launch a programmatic dependent of the
// previous one that is released as soon as its predecessor has READ its actions: chunk k+1's
// action reads (host -> GPU) then overlap chunk k's observation writes (GPU -> host); a single
// launch does all its reads first and all its writes last (measured, C1 at 4096 envs: 66 us per
// step in one launch = 18 compute + 17 reads + 27 writes, nothing overlapping).
static int zero_copy_chunks(const pgw_env* env) {
  if (!use_fused(env)) return 1;
  // (measured: a chain of chunks pays ~10 us per link for its own reads; staggering the tiles of
  // ONE launch gets the overlap without it.  The chain stays available as an option.)
  return env->host_chunks > 0 ? std::min(env->host_chunks, pgw_env::kMaxChunks) : 1;
}

// float32 actions: 128-byte rows.  Measured on a B200 (1000 W), C1 at 4096 envs, zero-copy step_host, wall us
// per call (medians of three sessions): 3 cycles per row 51.0, 2: 51.2, 5: 53.0, 10: 57.9, 0: 54.9
// (profiles/r4_e2e_io_dtype.jsonl, DESIGN.md section 6.0b)
constexpr int kStaggerPerRowF32 = 3;

static int enqueue_zero_copy(pgw_env* env, const void* actions, void* obs, double* rew, uint8_t* done,
                             bool io32, cudaStream_t s) {
  const int E = env->E, nch = zero_copy_chunks(env);
  // one tile's actions (act_dim x 256 B) at ~48 GB/s of PCIe reads, in cycles of the 1.965 GHz SM clock
  int per_row = io32 ? kStaggerPerRowF32 : 10;
  if (const char* v = getenv("PGW_STAGGER_CYCLES_PER_ROW")) per_row = atoi(v);   // tuning knob
  const int stagger = env->act_dim * per_row;
  if (nch == 1) return enqueue_step(env, actions, obs, rew, done, io32, s, false, 0, -1, 1, 0u, stagger);
  int bounds[pgw_env::kMaxChunks + 1];
  const int per = ((E + nch - 1) / nch + 31) / 32 * 32;             // whole 32-env tiles
  for (int k = 0; k <= nch; ++k) bounds[k] = std::min(E, k * per);
  unsigned int tickets = 0;
  for (int k = 0; k < nch; ++k)
    if (bounds[k + 1] > bounds[k]) tickets += (unsigned int)fused_grid(bounds[k + 1] - bounds[k]);
  bool first = true;
  for (int k = 0; k < nch; ++k) {
    if (bounds[k + 1] <= bounds[k]) continue;
    pgw::FusedParams P = step_fused_params(env, actions, obs, rew, done, io32, bounds[k], bounds[k + 1], tickets);
    P.pdl_trigger = 1;
    PGW_CUDA(pgw::launch_step_fused(P, fused_grid(bounds[k + 1] - bounds[k]), s, !first));
    first = false;
  }
  return PGW_OK;
}

static int zero_copy_step(pgw_env* env, const void* actions, void* obs, double* rew, uint8_t* done, bool io32,
                          cudaStream_t s) {
  const int nch = zero_copy_chunks(env);
  if (env->clock < 0) return fail(PGW_ERR_STATE, "pgw_step before pgw_reset");
  if (env->clock + 1 >= env->num_events) return fail(PGW_ERR_STATE, "episode is over: call pgw_reset");
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  PGW_CUDA(cudaStreamIsCapturing(s, &cap));
  cudaGraphExec_t exec = nullptr;
  if (env->use_graphs && cap == cudaStreamCaptureStatusNone && s != nullptr) {
    for (auto& g : env->host_graphs)
      if (g.actions == actions && g.obs == obs && g.rew == rew && g.done == done && g.io32 == io32) exec = g.exec;
    if (!exec && env->host_graphs.size() < 8) {        // a few pinned buffer sets; beyond: direct
      cudaGraph_t graph = nullptr;
      PGW_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      int rc = enqueue_zero_copy(env, actions, obs, rew, done, io32, s);
      cudaError_t ce = cudaStreamEndCapture(s, &graph);
      if (rc != PGW_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
      if (ce != cudaSuccess) return fail(PGW_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce));
      ce = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ce != cudaSuccess) return fail(PGW_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce));
      env->host_graphs.push_back({actions, obs, rew, done, io32, exec});
      ++env->graph_captures;
    }
  }
  if (exec) {
    PGW_CUDA(cudaGraphLaunch(exec, s));
  } else {
    int rc = enqueue_zero_copy(env, actions, obs, rew, done, io32, s);
    if (rc) return rc;
  }
  env->launches += nch * step_kernels(env);
  ++env->clock;
  return PGW_OK;
}

static int step_host_impl(pgw_env* env, const void* actions, void* obs, double* rew, uint8_t* done, bool io32,
                          void* cuda_stream) {
  if (!env || !actions || !obs || !rew || !done) return fail(PGW_ERR_INVALID, "null argument");
  if (env->clock < 0) return fail(PGW_ERR_STATE, "pgw_step before pgw_reset");
  if (env->clock + 1 >= env->num_events)
    return fail(PGW_ERR_STATE, "episode is over: call pgw_reset");
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  int rc;
  if (env->host_zero_copy && !env->timing) {
    // Page-locked host buffers: the kernels read the actions and write the observations,
    // rewards and done flags in place over PCIe (coalesced 256-byte requests; reads and posted
    // writes of different CTAs overlap in both directions of the link) -- no staging copies,
    // none of their ~8 us of fixed latency each.
    void* da = device_view(env, actions);
    void* dobs = device_view(env, obs);
    void* dr = device_view(env, rew);
    void* dd = device_view(env, done);
    if (da && dobs && dr && dd) {
      rc = zero_copy_step(env, da, dobs, static_cast<double*>(dr), static_cast<uint8_t*>(dd), io32, s);
      if (rc) return rc;
      PGW_CUDA(cudaStreamSynchronize(s));
      return PGW_OK;
    }
  }
  rc = ensure_staging(env, io32);
  if (rc) return rc;
  if (!env->ev_fork) {
    PGW_CUDA(cudaEventCreateWithFlags(&env->ev_fork, cudaEventDisableTiming));
    for (int k = 0; k < pgw_env::kMaxChunks; ++k) {
      PGW_CUDA(cudaStreamCreateWithFlags(&env->chunk_stream[k], cudaStreamNonBlocking));
      PGW_CUDA(cudaEventCreateWithFlags(&env->ev_join[k], cudaEventDisableTiming));
    }
  }
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  PGW_CUDA(cudaStreamIsCapturing(s, &cap));
  const bool graphable = env->use_graphs && !env->timing && cap == cudaStreamCaptureStatusNone &&
                         s != nullptr;
  cudaGraphExec_t exec = nullptr;
  if (graphable) {
    for (auto& g : env->host_graphs)
      if (g.actions == actions && g.obs == obs && g.rew == rew && g.done == done && g.io32 == io32) exec = g.exec;
    if (!exec && env->host_graphs.size() < 8) {        // a few pinned buffer sets; beyond: direct
      cudaGraph_t graph = nullptr;
      PGW_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      rc = enqueue_host_step(env, actions, obs, rew, done, io32, s);
      cudaError_t ce = cudaStreamEndCapture(s, &graph);
      if (rc != PGW_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
      if (ce != cudaSuccess) return fail(PGW_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce));
      ce = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ce != cudaSuccess) return fail(PGW_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce));
      env->host_graphs.push_back({actions, obs, rew, done, io32, exec});
      ++env->graph_captures;
    }
  }
  if (exec) {
    PGW_CUDA(cudaGraphLaunch(exec, s));
  } else if ((rc = enqueue_host_step(env, actions, obs, rew, done, io32, s))) {
    return rc;
  }
  PGW_CUDA(cudaStreamSynchronize(s));
  env->launches += step_kernels(env) * host_chunks(env, io32);
  ++env->clock;
  return PGW_OK;
}

int pgw_step_host(pgw_env* env, const double* actions, double* obs, double* rew, uint8_t* done,
                  void* cuda_stream) {
  return step_host_impl(env, actions, obs, rew, done, false, cuda_stream);
}

int pgw_step_host_f32(pgw_env* env, const float* actions, float* obs, double* rew, uint8_t* done,
                      void* cuda_stream) {
  return step_host_impl(env, actions, obs, rew, done, true, cuda_stream);
}

static int field_location(pgw_env* env, int field, void** ptr, size_t* want) {
  const size_t E = (size_t)env->E, A = (size_t)env->A;
  switch (field) {
    case PGW_FIELD_STATE_D: *ptr = env->sd; *want = (size_t)env->sd_rows * E * 8; break;
    case PGW_FIELD_STATE_I: *ptr = env->si; *want = (size_t)env->si_rows * E * 4; break;
    case PGW_FIELD_AGENT_P: *ptr = env->agent_p; *want = A * E * 8; break;
    case PGW_FIELD_VOLTAGES: *ptr = env->vmag; *want = (size_t)env->pf_base.nn * E * 8; break;
    case PGW_FIELD_VMIN: *ptr = env->vmin; *want = E * 8; break;
    case PGW_FIELD_VMAX: *ptr = env->vmax; *want = E * 8; break;
    case PGW_FIELD_VBUS: *ptr = env->vbus; *want = A * E * 8; break;
    case PGW_FIELD_PF_ITERS: *ptr = env->iters; *want = E * 4; break;
    case PGW_FIELD_EP_RETURN: *ptr = env->ep_ret; *want = A * E * 8; break;
    case PGW_FIELD_PF_STATE: *ptr = env->u_state; *want = (size_t)env->pf_base.nbp * E * 16; break;
    default: return fail(PGW_ERR_INVALID, "unknown field");
  }
  return PGW_OK;
}

static int check_size(size_t want, size_t bytes) {
  if (bytes == want) return PGW_OK;
  char buf[128];
  snprintf(buf, sizeof buf, "size mismatch: field needs %zu bytes, got %zu", want, bytes);
  return fail(PGW_ERR_INVALID, buf);
}

int pgw_get(pgw_env* env, int field, void* dst, size_t bytes, void* cuda_stream) {
  if (!env || !dst) return fail(PGW_ERR_INVALID, "null argument");
  void* src = nullptr;
  size_t want = 0;
  int rc = field_location(env, field, &src, &want);
  if (rc) return rc;
  if (want == 0) return PGW_OK;
  if (!src) return fail(PGW_ERR_INVALID, "field not available (no feeder)");
  if ((rc = check_size(want, bytes))) return rc;
  PGW_CUDA(cudaMemcpyAsync(dst, src, want, cudaMemcpyDeviceToDevice,
                           static_cast<cudaStream_t>(cuda_stream)));
  return PGW_OK;
}

int pgw_set(pgw_env* env, int field, const void* src, size_t bytes, void* cuda_stream) {
  if (!env || !src) return fail(PGW_ERR_INVALID, "null argument");
  void* dst = nullptr;
  size_t want = 0;
  int rc = field_location(env, field, &dst, &want);
  if (rc) return rc;
  if (want == 0) return PGW_OK;
  if (!dst) return fail(PGW_ERR_INVALID, "field not available (no feeder)");
  if ((rc = check_size(want, bytes))) return rc;
  PGW_CUDA(cudaMemcpyAsync(dst, src, want, cudaMemcpyDeviceToDevice,
                           static_cast<cudaStream_t>(cuda_stream)));
  return PGW_OK;
}

int pgw_set_rows(pgw_env* env, int field, int row_begin, int row_count, const void* src, size_t bytes,
                 void* cuda_stream) {
  if (!env || !src) return fail(PGW_ERR_INVALID, "null argument");
  if (field != PGW_FIELD_STATE_D && field != PGW_FIELD_STATE_I)
    return fail(PGW_ERR_INVALID, "pgw_set_rows serves the two state arrays");
  const int rows = field == PGW_FIELD_STATE_D ? env->sd_rows : env->si_rows;
  const size_t el = field == PGW_FIELD_STATE_D ? 8 : 4;
  if (row_begin < 0 || row_count < 0 || row_begin + row_count > rows)
    return fail(PGW_ERR_INVALID, "row range outside the field");
  int rc = check_size((size_t)row_count * (size_t)env->E * el, bytes);
  if (rc) return rc;
  if (row_count == 0) return PGW_OK;
  unsigned char* base = field == PGW_FIELD_STATE_D ? reinterpret_cast<unsigned char*>(env->sd)
                                                   : reinterpret_cast<unsigned char*>(env->si);
  PGW_CUDA(cudaMemcpyAsync(base + (size_t)row_begin * (size_t)env->E * el, src, bytes, cudaMemcpyDeviceToDevice,
                           static_cast<cudaStream_t>(cuda_stream)));
  return PGW_OK;
}

int pgw_set_clock(pgw_env* env, int steps, void* cuda_stream) {
  if (!env) return fail(PGW_ERR_INVALID, "null argument");
  if (steps < 0 || steps >= env->num_events) return fail(PGW_ERR_INVALID, "clock out of range");
  PGW_CUDA(cudaMemcpyAsync(env->d_clock, &steps, sizeof(int), cudaMemcpyHostToDevice,
                           static_cast<cudaStream_t>(cuda_stream)));
  PGW_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(cuda_stream)));
  env->clock = steps;
  return PGW_OK;
}

int pgw_update_tables(pgw_env* env, const double* dpar, int dpar_len, const double* dtab,
                      const int32_t* itab, void* cuda_stream) {
  if (!env) return fail(PGW_ERR_INVALID, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  if (dpar) {
    if (dpar_len != env->dpar_len) return fail(PGW_ERR_INVALID, "parameter block length changed");
    if (dpar_len)
      PGW_CUDA(cudaMemcpyAsync(env->comp_blob + env->comp_base.off_dpar, dpar, (size_t)dpar_len * sizeof(double),
                               cudaMemcpyHostToDevice, s));
  }
  if (dtab)
    PGW_CUDA(cudaMemcpyAsync(env->dtab, dtab, (size_t)env->num_events * env->comp_base.dstride * sizeof(double),
                             cudaMemcpyHostToDevice, s));
  if (itab && env->comp_base.istride)
    PGW_CUDA(cudaMemcpyAsync(env->itab, itab, (size_t)env->num_events * env->comp_base.istride * sizeof(int32_t),
                             cudaMemcpyHostToDevice, s));
  PGW_CUDA(cudaStreamSynchronize(s));
  return PGW_OK;
}

int pgw_pf_solve(pgw_env* env, const double* load_kw, const double* load_kvar,
                 void* cuda_stream) {
  if (!env || !load_kw || !load_kvar) return fail(PGW_ERR_INVALID, "null argument");
  if (!env->has_feeder) return fail(PGW_ERR_INVALID, "this env has no feeder");
  pgw::PfParams pf = env->pf_base;
  pf.event_mode = 0; pf.advance_clock = 0; pf.agent_p = nullptr; pf.rew = nullptr;
  pf.punit = 0.0; pf.load_kw = load_kw; pf.load_kvar = load_kvar; pf.warm_start = 0;
  PGW_CUDA(launch_pf(env, pf, static_cast<cudaStream_t>(cuda_stream)));
  ++env->launches;
  return PGW_OK;
}

int pgw_stats(pgw_env* env, double* out, void* cuda_stream) {
  if (!env || !out) return fail(PGW_ERR_INVALID, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  static const double init[PGW_NUM_STATS] = {0, 0, 0, 0, 0, 0, 1e300, 0};
  PGW_CUDA(cudaMemcpyAsync(out, init, sizeof init, cudaMemcpyHostToDevice, s));
  pgw::StatsParams p{};
  p.E = env->E; p.A = env->A; p.nn = env->pf_base.nn;
  p.rew = env->rew_last; p.ep_ret = env->ep_ret;
  p.viol = env->viol; p.iters = env->has_feeder ? env->iters : nullptr;
  p.vmin = env->vmin; p.vmax = env->vmax; p.clock = env->d_clock; p.out = out;
  PGW_CUDA(pgw::launch_stats(p, s));
  ++env->launches;
  return PGW_OK;
}

int pgw_set_timing(pgw_env* env, int enabled) {
  if (!env) return fail(PGW_ERR_INVALID, "null argument");
  env->timing = enabled != 0;
  env->ev_used = 0;
  env->t_comp_ms = env->t_pf_ms = env->t_steps = 0;
  return PGW_OK;
}

int pgw_get_timing(pgw_env* env, double* out3, void* cuda_stream) {
  if (!env || !out3) return fail(PGW_ERR_INVALID, "null argument");
  PGW_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(cuda_stream)));
  for (size_t i = 0; i + 2 < env->ev_used; i += 3) {
    float a = 0, b = 0;
    PGW_CUDA(cudaEventElapsedTime(&a, env->ev_pool[i], env->ev_pool[i + 1]));
    PGW_CUDA(cudaEventElapsedTime(&b, env->ev_pool[i + 1], env->ev_pool[i + 2]));
    env->t_comp_ms += a;
    env->t_pf_ms += b;
    env->t_steps += 1;
  }
  env->ev_used = 0;
  out3[0] = env->t_comp_ms; out3[1] = env->t_pf_ms; out3[2] = env->t_steps;
  env->t_comp_ms = env->t_pf_ms = env->t_steps = 0;
  return PGW_OK;
}

int pgw_clock(const pgw_env* env) { return env ? env->clock : -1; }

#ifdef PGW_PHASE_TIMERS
// instrumented builds only: SM-clock stamps of the power-flow kernel's phases, [ctas][16]
int pgw_debug_phases(pgw_env* env, long long* host_out, int ctas) {
  if (!env || !host_out || ctas > 4096) return PGW_ERR_INVALID;
  PGW_CUDA(cudaDeviceSynchronize());
  PGW_CUDA(cudaMemcpy(host_out, env->phase_clk, (size_t)ctas * 16 * sizeof(long long),
                      cudaMemcpyDeviceToHost));
  return PGW_OK;
}
// component kernel CTAs, [ctas][8]: globaltimer at entry / exit, then SM-clock phase stamps
int pgw_debug_comp_span(pgw_env* env, long long* host_out, int ctas) {
  if (!env || !host_out || ctas > 4096) return PGW_ERR_INVALID;
  PGW_CUDA(cudaDeviceSynchronize());
  PGW_CUDA(cudaMemcpy(host_out, env->phase_clk + (size_t)4096 * 16,
                      (size_t)ctas * 8 * sizeof(long long), cudaMemcpyDeviceToHost));
  return PGW_OK;
}
#endif
// CTAs of the component kernel's CTA table (tests check it against a mirror of the allocation)
int pgw_debug_num_comp_ctas(pgw_env* env) { return env ? env->comp_base.num_ctas : 0; }
long long pgw_launch_count(const pgw_env* env) { return env ? env->launches : 0; }
long long pgw_graph_captures(const pgw_env* env) { return env ? env->graph_captures : 0; }
long long pgw_reset_count(const pgw_env* env) { return env ? env->resets : 0; }
int pgw_set_reset_count(pgw_env* env, long long resets) {
  if (!env || resets < 0) return fail(PGW_ERR_INVALID, "invalid argument");
  env->resets = resets;
  return PGW_OK;
}

int pgw_set_option(pgw_env* env, int option, int value) {
  if (env && option == PGW_OPT_CLIP_INIT_SOC) {      // a reset parameter: the step graphs stay valid
    env->clip_init_soc = value != 0;
    return PGW_OK;
  }
  if (!env) return fail(PGW_ERR_INVALID, "null argument");
  switch (option) {
    case PGW_OPT_PF_KERNEL:
      if (value < 0 || value > 2) return fail(PGW_ERR_INVALID, "unknown power-flow kernel");
      if (value == 2 && !env->pf_base.tc2.blob)
        return fail(PGW_ERR_INVALID, "FP16 tensor-core power flow needs a feeder with <= 88 load "
                                     "branches whose tables fit shared memory");
      if (value == 1 && !env->pf_base.tc_blob)
        return fail(PGW_ERR_INVALID, "tensor-core power flow needs a feeder with <= 16 load "
                                     "branches and <= 48 nodes");
      env->pf_kernel = value;
      break;
    case PGW_OPT_WARM_START: env->warm_start = value != 0; break;
    case PGW_OPT_GRAPHS: env->use_graphs = value != 0; break;
    case PGW_OPT_PDL: env->use_pdl = value != 0; break;
    case PGW_OPT_HOST_ZERO_COPY: env->host_zero_copy = value != 0; break;
    case PGW_OPT_HOST_CHUNKS:
      if (value < 0 || value > pgw_env::kMaxChunks) return fail(PGW_ERR_INVALID, "0 (automatic) .. 8 chunks");
      env->host_chunks = value;
      break;
    case PGW_OPT_FUSED:
      if (value < 0 || value > 2) return fail(PGW_ERR_INVALID, "PGW_OPT_FUSED takes 0, 1 or 2");
      if (value == 2 && !env->fused_ok)
        return fail(PGW_ERR_INVALID, "the fused step kernel does not serve this scenario");
      env->fused_mode = value;
      break;
    case PGW_OPT_PF_POLISH:
      if (value < 0 || value > 8) return fail(PGW_ERR_INVALID, "polish sweeps out of range (0..8)");
      if (value > 0 && !env->pf_base.tc2.polish_ok)
        return fail(PGW_ERR_INVALID, "the FP64 polish serves feeders with <= 16 load branches");
      env->pf_base.tc2.polish = value;
      if (!env->tc2_tol_set) env->pf_base.tc2.tol = pgw::tc2_default_tol(env->pf_base.tol, value);
      break;
    case PGW_OPT_PF_TC_TOL_NANO:
      if (value < 10 || value > 100000) return fail(PGW_ERR_INVALID, "tolerance out of range (1e-8..1e-4)");
      env->pf_base.tc2.tol = (float)(value * 1e-9);
      env->tc2_tol_set = true;
      break;
    default: return fail(PGW_ERR_INVALID, "unknown option");
  }
  // the captured graphs bake the options in
  env->drop_graphs();
  return PGW_OK;
}

}  // extern "C"
