// C ABI of the batched simulator (include/pgw.h): owns the device-side tables and
// state of one env batch and sequences the kernels of reset / step.
//
//   reset:  [power flow, base load only]  ->  [component reset kernel]
//   step:   [component step kernel]       ->  [power flow + reward hook]
//
// The episode clock lives on the device and is advanced by the last CTA of the last
// kernel of a step, so a step has constant launch parameters (CUDA-graph friendly).
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "internal.cuh"

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

int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Convergence threshold max|d drop| (p.u.) of the tcgen05 fixed point.  The float32 iteration cannot
// resolve less than ~1e-7.  Where the float64 polish follows (its two sweeps contract whatever the loop
// leaves behind by > 100x for the voltages the rewards read) the loop stops at 1e-6: one iteration
// less per solve, rewards and voltages unchanged within their bounds (measured over 2.3 M env-steps:
// worst reward error 0.093 of the bound against 0.089 at 1e-7, node voltages 2.3e-7 p.u. either way;
// tools/reward_margin.py).  OpenDSS's own convergence tolerance is 1e-4.
float tc2_default_tol(double solver_tol, int polish) {
  const double floor_tol = polish > 0 ? 1e-6 : 1e-7;
  return (float)(solver_tol > floor_tol ? solver_tol : floor_tol);
}

}  // namespace

struct pgw_env {
  int E = 0, A = 0, C = 0, act_dim = 0, obs_dim = 0, sd_rows = 0, si_rows = 0;
  int num_storage = 0, num_events = 0, dstride = 0, istride = 0;
  bool has_feeder = false;
  bool need_scratch = false, need_scratch_reset = false;
  int nb = 0, nn = 0, nl = 0, nbp = 0, nnp = 0, max_iter = 0;
  double tol = 0;
  int penalty_node = -1;
  double pvlo = 0, pvhi = 0, punit = 0;
  int pf_kernel = 0;
  int clock = -1;             // host mirror
  long long resets = 0;
  int has_house = 0;          // 1 = houses, 2 = houses with step_meta telemetry
  bool ev_per_env = false;    // some charging station runs on per-env rosters (PGW_F_EV_PER_ENV)
  long long launches = 0;
  long long graph_captures = 0;        // graphs captured + instantiated since creation
  // device tables
  unsigned char* comp_blob = nullptr;   // [agents | comps | dpar | ipar]
  int comp_blob_bytes = 0, off_comps = 0, off_dpar = 0, off_ipar = 0, dpar_len = 0;
  pgw::CtaWork* work = nullptr;         // CTA -> (agent, env blocks, staging ranges)
  int num_ctas = 0;
  int max_cn = 0, max_dn = 0, max_in = 0;
  double* dtab = nullptr;
  int32_t* itab = nullptr;
  unsigned char* pf_blob = nullptr;     // feeder tables, layout in internal.cuh
  int pf_blob_bytes = 0, pf_stage = 0;
  int off_u0 = 0, off_znbT = 0, off_w = 0, off_share = 0, off_vmin = 0, off_vmax = 0,
      off_bload = 0, off_bmodel = 0, off_slot = 0, off_node = 0;
  double2* u_state = nullptr;
  bool warm_start = true;
  // tensor-core power flow (powerflow_tc.cu): operand images + fp32 tables
  unsigned char* tc_blob = nullptr;
  int tc_blob_bytes = 0, tc_n2 = 0, tc_nnp8 = 0;
  int tc_off_b2 = 0, tc_off_u0 = 0, tc_off_w = 0, tc_off_share = 0, tc_off_vlo = 0, tc_off_vhi = 0,
      tc_off_bload = 0, tc_off_bmodel = 0, tc_off_slot = 0, tc_off_node = 0;
  // FP16 tensor-core power flow for up to 88 load branches (powerflow_tc2.cu)
  unsigned char* tc2_blob = nullptr;
  pgw::Tc2Params tc2{};
  bool tc2_tol_set = false;             // PGW_OPT_PF_TC_TOL_NANO was given: the polish option leaves tol alone
  pgw::Tc2Consts tc2c{};
  pgw::Tc2Polish tc2p{};
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
  if (spec->abi_version != PGW_ABI_VERSION) return fail(PGW_ERR_INVALID, "ABI version mismatch");
  if (spec->num_envs <= 0 || spec->num_agents <= 0 || spec->num_components <= 0 ||
      spec->num_events <= 1)
    return fail(PGW_ERR_INVALID, "empty spec");
  if (spec->dtab_stride % 2 || spec->itab_stride % 4)
    return fail(PGW_ERR_INVALID, "event rows must be multiples of 16 bytes");
  if (spec->num_agents > 65535) return fail(PGW_ERR_INVALID, "too many agents");
  for (int a = 0; a < spec->num_agents; ++a) {
    const pgw_agent& ag = spec->agents[a];
    if (ag.comp_begin < 0 || ag.comp_end > spec->num_components || ag.comp_begin >= ag.comp_end)
      return fail(PGW_ERR_INVALID, "agent component range out of bounds");
    if (ag.load_slot >= 0 && (!spec->feeder || ag.load_slot >= spec->feeder->nl))
      return fail(PGW_ERR_INVALID, "agent load slot out of range");
    if (ag.bus_node >= 0 && (!spec->feeder || ag.bus_node >= spec->feeder->nn))
      return fail(PGW_ERR_INVALID, "agent bus node out of range");
  }
  for (int c = 0; c < spec->num_components; ++c) {
    const pgw_component& k = spec->components[c];
    if (k.type < PGW_STORAGE || k.type > PGW_HS_DEVICES)
      return fail(PGW_ERR_INVALID, "unknown component type (no CPU fallback exists)");
    if (k.obs_off < 0 || k.obs_off + k.obs_dim > spec->obs_dim || k.act_off < 0 ||
        k.act_off >= spec->act_dim || k.dpar_off < 0 || k.dpar_off > spec->dpar_len ||
        k.ipar_off < 0 || k.ipar_off > spec->ipar_len)
      return fail(PGW_ERR_INVALID, "component offsets out of range");
    {
      // rows each component kind reads and writes (layouts in include/pgw.h): a spec that is off
      // by a row must come back as PGW_ERR_INVALID, not as an out-of-bounds access on the device
      auto ip = [&](int i) { return k.ipar_off + i < spec->ipar_len ? spec->ipar[k.ipar_off + i] : -1; };
      const bool tel = (k.flags & PGW_F_TELEMETRY) != 0;
      int act = 1, obs_min = 1, sd = 0, si = 0, dw = 0, iw = 0;
      switch (k.type) {
        case PGW_STORAGE: sd = 1; break;
        case PGW_PV: obs_min = (k.flags & PGW_F_GRID_AWARE) ? 2 : 1; dw = 1; break;
        case PGW_EV: case PGW_HS_EV: {
          const int n = ip(0), words = ip(1), cap = ip(2);
          if (k.flags & PGW_F_EV_PER_ENV) {            // per-env rosters: window words behind the mask
            if (k.type != PGW_EV || n <= 0 || n > 256 || words != (n + 31) / 32)
              return fail(PGW_ERR_INVALID, "EV station with per-env rosters: stock station, 1..256 vehicles, "
                                           "ipar = n, ceil(n/32), 0");
            obs_min = 6; sd = n; si = words + n; dw = 2; iw = 0;
            break;
          }
          if (n <= 0 || words != (n + 31) / 32 || cap <= 0)
            return fail(PGW_ERR_INVALID, "EV station: ipar must hold n, ceil(n/32), list capacity");
          obs_min = k.type == PGW_EV ? 6 : 7;
          sd = n + (k.type == PGW_HS_EV ? 1 : 0); si = words; dw = 2 + 2 * cap; iw = 2 + 2 * cap;
          break;
        }
        case PGW_BUILDING: act = 6; sd = 6; dw = 17; break;
        case PGW_HS_BEGIN: act = 0; obs_min = 0; sd = 5; dw = 1; break;
        case PGW_HS_PV: dw = 1; break;
        case PGW_HS_STORAGE: obs_min = 2; sd = 2; break;
        case PGW_HS_DEVICES: {
          const int cols = ip(0);
          if (cols <= 0) return fail(PGW_ERR_INVALID, "devices: ipar must hold the column count");
          obs_min = cols; dw = 2 * cols;
          break;
        }
        default: break;
      }
      if (tel && k.type >= PGW_HS_PV) sd += PGW_HS_TEL_ROWS;
      if (k.act_off + act > spec->act_dim) return fail(PGW_ERR_INVALID, "component action rows out of range");
      if (k.obs_dim < obs_min) return fail(PGW_ERR_INVALID, "component observation rows: fewer than the kind writes");
      if (k.sd_off < 0 || k.sd_off + sd > spec->sd_rows || k.si_off < 0 || k.si_off + si > spec->si_rows)
        return fail(PGW_ERR_INVALID, "component state rows out of range");
      if (k.dtab_off < 0 || k.dtab_off + dw > spec->dtab_stride || k.itab_off < 0 ||
          k.itab_off + iw > spec->itab_stride)
        return fail(PGW_ERR_INVALID, "component event-row block out of range");
    }
    if (!spec->feeder && (k.flags & (PGW_F_GRID_AWARE | PGW_F_PV_VOLT_REWARD)))
      return fail(PGW_ERR_INVALID, "grid-aware component without a feeder");
    if (k.type == PGW_BUILDING && (k.flags & PGW_F_BUILDING_FAST) && k.obs_dim != 15)
      return fail(PGW_ERR_INVALID, "PGW_F_BUILDING_FAST requires the 15-entry observation set");
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
  env->num_storage = spec->num_storage; env->num_events = spec->num_events;
  env->dstride = spec->dtab_stride; env->istride = spec->itab_stride;
  for (int c = 0; c < spec->num_components; ++c) {
    if (spec->components[c].type == PGW_HS_BEGIN) env->has_house = std::max(env->has_house, 1);
    if (spec->components[c].flags & PGW_F_EV_PER_ENV) env->ev_per_env = true;
  }
  for (int c = 0; c < spec->num_components; ++c)
    if (spec->components[c].type >= PGW_HS_PV && (spec->components[c].flags & PGW_F_TELEMETRY))
      env->has_house = 2;
  for (int c = 0; c < spec->num_components; ++c)
    if (spec->components[c].type == PGW_BUILDING) {
      env->need_scratch_reset = true;                // reset always takes the table-driven path
      if (!(spec->components[c].flags & PGW_F_BUILDING_FAST)) env->need_scratch = true;
    }
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

  {
    // static component tables as one blob, staged to shared memory by every CTA
    const size_t b_ag = A * sizeof(pgw_agent);
    const size_t b_co = (size_t)env->C * sizeof(pgw_component);
    const size_t b_dp = (size_t)spec->dpar_len * sizeof(double);
    const size_t b_ip = (size_t)spec->ipar_len * sizeof(int32_t);
    env->dpar_len = spec->dpar_len;
    env->off_comps = round_up((int)b_ag, 16);
    env->off_dpar = round_up(env->off_comps + (int)b_co, 16);
    env->off_ipar = round_up(env->off_dpar + (int)b_dp, 16);
    env->comp_blob_bytes = round_up(env->off_ipar + (int)b_ip, 16);
    std::vector<unsigned char> blob(env->comp_blob_bytes, 0);
    memcpy(blob.data(), spec->agents, b_ag);
    memcpy(blob.data() + env->off_comps, spec->components, b_co);
    if (b_dp) memcpy(blob.data() + env->off_dpar, spec->dpar, b_dp);
    if (b_ip) memcpy(blob.data() + env->off_ipar, spec->ipar, b_ip);
    PGW_TRY(upload(&env->comp_blob, blob.data(), blob.size())); env->own(env->comp_blob);
    // per-agent slices: components [begin, end), and the span of their parameter blocks (a
    // block ends where the next larger offset of any component starts)
    std::vector<int> dstart, istart;
    for (int c = 0; c < env->C; ++c) {
      dstart.push_back(spec->components[c].dpar_off);
      istart.push_back(spec->components[c].ipar_off);
    }
    dstart.push_back(spec->dpar_len); istart.push_back(spec->ipar_len);
    std::sort(dstart.begin(), dstart.end()); std::sort(istart.begin(), istart.end());
    auto block_end = [](const std::vector<int>& starts, int off) {
      return *std::upper_bound(starts.begin(), starts.end(), off);
    };
    std::vector<pgw::AgentSlice> sl(env->A);
    for (int a = 0; a < env->A; ++a) {
      const pgw_agent& ag = spec->agents[a];
      int dlo = spec->dpar_len, dhi = 0, ilo = spec->ipar_len, ihi = 0;
      for (int c = ag.comp_begin; c < ag.comp_end; ++c) {
        const pgw_component& k = spec->components[c];
        if (k.dpar_off < spec->dpar_len) {
          dlo = std::min(dlo, k.dpar_off); dhi = std::max(dhi, block_end(dstart, k.dpar_off));
        }
        if (k.ipar_off < spec->ipar_len) {
          ilo = std::min(ilo, k.ipar_off); ihi = std::max(ihi, block_end(istart, k.ipar_off));
        }
      }
      if (dhi <= dlo) dlo = dhi = 0;
      if (ihi <= ilo) ilo = ihi = 0;
      pgw::AgentSlice& s = sl[a];
      s.c_lo = ag.comp_begin; s.c_n = ag.comp_end - ag.comp_begin;
      s.d_lo = dlo / 2 * 2; s.d_n = round_up(dhi - s.d_lo, 2);
      s.i_lo = ilo / 4 * 4; s.i_n = round_up(ihi - s.i_lo, 4);
      s.pad0 = s.pad1 = 0;
      env->max_cn = std::max(env->max_cn, s.c_n);
      env->max_dn = std::max(env->max_dn, s.d_n);
      env->max_in = std::max(env->max_in, s.i_n);
    }
    // CTA budget of ~16 per SM, split over the agents in proportion to a cost estimate of their
    // components (rough time per 64-env block), every agent between 1 CTA and one CTA per
    // 64-env block.
    {
      // 16 CTAs per SM (10 are resident: 96 registers x 64 threads) lets the hardware scheduler
      // even out the rough cost estimates of a many-agent scenario (C3: 134 us at 16 per SM,
      // 150 us at 10); with a single agent there is nothing to even out and a second round of
      // CTAs only adds a partial wave (262 144 houses: 42.3 us at 16 per SM, 35.8 us at 10).
      int budget = env->A == 1 ? 148 * 10 : 148 * 16;
      if (const char* b = getenv("PGW_CTA_BUDGET")) budget = std::max(1, atoi(b));   // tuning knob
      const int blocks = (env->E + 63) / 64;
      std::vector<double> w(env->A, 0.5);            // ~us per env block: loop + latency floor
      double wsum = 0.0;
      for (int a = 0; a < env->A; ++a) {
        for (int c = spec->agents[a].comp_begin; c < spec->agents[a].comp_end; ++c) {
          const pgw_component& k = spec->components[c];
          switch (k.type) {
            case PGW_BUILDING: w[a] += 2.0; break;
            case PGW_EV: case PGW_HS_EV: w[a] += 1.0 + 0.04 * spec->ipar[k.ipar_off]; break;
            case PGW_STORAGE: w[a] += 0.8; break;
            case PGW_HS_BEGIN: case PGW_HS_STORAGE: case PGW_HS_DEVICES: w[a] += 1.0; break;
            default: w[a] += 0.5; break;
          }
        }
        wsum += w[a];
      }
      // water-filling: agents that reach one CTA per block give their surplus to the others
      std::vector<int> n(env->A, 0);
      {
        std::vector<char> capped(env->A, 0);
        double left = budget, wleft = wsum;
        for (bool again = true; again;) {
          again = false;
          for (int a = 0; a < env->A; ++a)
            if (!capped[a] && left * w[a] / wleft >= blocks) {
              capped[a] = 1; n[a] = blocks; left -= blocks; wleft -= w[a]; again = true;
            }
        }
        for (int a = 0; a < env->A; ++a)
          if (!capped[a])
            n[a] = std::max(1, std::min(blocks, (int)std::ceil(left * w[a] / wleft)));
      }
      std::vector<int> order(env->A);
      for (int a = 0; a < env->A; ++a) order[a] = a;
      std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return w[x] > w[y]; });
      // longest-processing-time-first: every CTA of the heaviest agent, then the next agent, ...
      // so that the long-running CTAs are all resident from the start and the light ones fill in
      // behind them (with round-robin emission half of an EV station's CTAs started a wave late)
      std::vector<pgw::CtaWork> work;
      for (int a : order)
        for (int j = 0; j < n[a]; ++j) {
          pgw::CtaWork cw{};
          cw.agent = a; cw.j = j; cw.n = n[a]; cw.sl = sl[a];
          work.push_back(cw);
        }
      env->num_ctas = (int)work.size();
      PGW_TRY(upload(&env->work, work.data(), work.size())); env->own(env->work);
    }
    if (env->max_cn * (int)sizeof(pgw_component) + env->max_dn * 8 + env->max_in * 4 +
            spec->dtab_stride * 8 + spec->itab_stride * 4 > 160 * 1024) {
      delete env;
      return fail(PGW_ERR_INVALID, "scenario tables exceed the shared-memory staging budget");
    }
  }
  PGW_TRY(upload(&env->dtab, spec->dtab, (size_t)spec->num_events * spec->dtab_stride));
  env->own(env->dtab);
  PGW_TRY(upload(&env->itab, spec->itab, (size_t)spec->num_events * spec->itab_stride));
  env->own(env->itab);

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

  if (spec->feeder) {
    const pgw_feeder& f = *spec->feeder;
    if (f.nb <= 0 || f.nn <= 0 || f.nl <= 0 || f.nb > 128 || f.max_iter <= 0) {
      delete env;
      return fail(PGW_ERR_INVALID, "feeder dimensions out of range (1..128 load branches)");
    }
    if (spec->dtab_stride < 2 + 2 * f.nl) {
      delete env;
      return fail(PGW_ERR_INVALID, "event row too short for the feeder base loads");
    }
    env->has_feeder = true;
    env->nb = f.nb; env->nn = f.nn; env->nl = f.nl; env->max_iter = f.max_iter; env->tol = f.tol;
    env->nbp = f.nb <= 16 ? 16 : round_up(f.nb, 32);
    env->nnp = round_up(f.nn, 2);
    env->penalty_node = f.penalty_node; env->pvlo = f.penalty_vlo; env->pvhi = f.penalty_vhi;
    env->punit = f.penalty_unit;
    if (env->punit != 0.0 && (f.penalty_node < 0 || f.penalty_node >= f.nn)) {
      delete env;
      return fail(PGW_ERR_INVALID, "penalty node out of range");
    }
    const int nb = f.nb, nn = f.nn, nbp = env->nbp, nnp = env->nnp;
    std::vector<double2> zt((size_t)nb * nbp, make_double2(0, 0)), u0(nbp, make_double2(1, 0)),
        znt((size_t)nb * nnp, make_double2(0, 0)), w(nnp, make_double2(0, 0));
    for (int k = 0; k < nb; ++k)
      for (int j = 0; j < nb; ++j)
        zt[(size_t)j * nbp + k] = make_double2(f.zbb[2 * ((size_t)k * nb + j)], f.zbb[2 * ((size_t)k * nb + j) + 1]);
    for (int k = 0; k < nb; ++k) u0[k] = make_double2(f.u0[2 * k], f.u0[2 * k + 1]);
    for (int n = 0; n < nn; ++n) {
      w[n] = make_double2(f.w[2 * n], f.w[2 * n + 1]);
      for (int k = 0; k < nb; ++k)
        znt[(size_t)k * nnp + n] = make_double2(f.znb[2 * ((size_t)n * nb + k)], f.znb[2 * ((size_t)n * nb + k) + 1]);
    }
    std::vector<int32_t> bl(nbp, 0), bm(nbp, 1);
    std::vector<double> bs(nbp, 0.0), vlo(nbp, 0.95), vhi(nbp, 1.05);
    for (int k = 0; k < nb; ++k) {
      if (f.branch_load[k] < 0 || f.branch_load[k] >= f.nl) {
        delete env;
        return fail(PGW_ERR_INVALID, "branch load index out of range");
      }
      bl[k] = f.branch_load[k]; bm[k] = f.branch_model[k]; bs[k] = f.branch_share[k];
      vlo[k] = f.vminpu[k]; vhi[k] = f.vmaxpu[k];
    }
    {
      std::vector<int32_t> slot(env->A), node(env->A);
      for (int a = 0; a < env->A; ++a) {
        slot[a] = spec->agents[a].load_slot;
        node[a] = spec->agents[a].bus_node;
      }
      std::vector<unsigned char> blob;
      auto put = [&blob](const void* src, size_t bytes) {
        const size_t off = (blob.size() + 15) / 16 * 16;
        blob.resize(off + bytes, 0);
        memcpy(blob.data() + off, src, bytes);
        return (int)off;
      };
      put(zt.data(), zt.size() * sizeof(double2));
      env->off_u0 = put(u0.data(), u0.size() * sizeof(double2));
      env->off_znbT = put(znt.data(), znt.size() * sizeof(double2));
      env->off_w = put(w.data(), w.size() * sizeof(double2));
      env->off_share = put(bs.data(), bs.size() * 8);
      env->off_vmin = put(vlo.data(), vlo.size() * 8);
      env->off_vmax = put(vhi.data(), vhi.size() * 8);
      env->off_bload = put(bl.data(), bl.size() * 4);
      env->off_bmodel = put(bm.data(), bm.size() * 4);
      env->off_slot = put(slot.data(), slot.size() * 4);
      env->off_node = put(node.data(), node.size() * 4);
      blob.resize((blob.size() + 15) / 16 * 16, 0);
      env->pf_blob_bytes = (int)blob.size();
      env->pf_stage = env->pf_blob_bytes <= 96 * 1024 ? 1 : 0;   // else read through L1/L2
      PGW_TRY(upload(&env->pf_blob, blob.data(), blob.size())); env->own(env->pf_blob);
    }
    PGW_TRY(alloc_zero(&env->u_state, (size_t)nbp * E)); env->own(env->u_state);
    if (nb <= pgw::kTcNb && 32 + 2 * round_up(nn, 8) <= 128) {
      // Operand images of the tcgen05 kernel, byte-exact as they sit in shared memory:
      // canonical K-major no-swizzle UMMA layout, element (row, k) at
      //   (row/8)*3072 + (k/4)*128 + (row%8)*16 + (k%4)*4,   K = 96 = [hi | hi | lo] of B.
      const int NB = pgw::kTcNb, K3 = pgw::kTcK3, nnp8 = round_up(nn, 8), n2 = 2 * nnp8;
      auto hi_of = [](double v) {
        float f = (float)v;
        uint32_t u;
        memcpy(&u, &f, 4);
        u &= 0xFFFFE000u;
        memcpy(&f, &u, 4);
        return f;
      };
      auto image = [&](int rows, const std::vector<double>& b /* [rows][32] */) {
        std::vector<unsigned char> img((size_t)rows * K3 * 4, 0);
        for (int r = 0; r < rows; ++r)
          for (int k = 0; k < 32; ++k) {
            const double v = b[(size_t)r * 32 + k];
            const float hi = hi_of(v), lo = (float)(v - (double)hi);
            const float part[3] = {hi, hi, lo};
            for (int q = 0; q < 3; ++q) {
              const int kc = q * 32 + k;
              const size_t off = (size_t)(r / 8) * 3072 + (size_t)(kc / 4) * 128 + (r % 8) * 16 + (kc % 4) * 4;
              memcpy(img.data() + off, &part[q], 4);
            }
          }
        return img;
      };
      auto Z = [&](int k, int j) { return make_double2(f.zbb[2 * ((size_t)k * nb + j)], f.zbb[2 * ((size_t)k * nb + j) + 1]); };
      auto ZN = [&](int n, int k) { return make_double2(f.znb[2 * ((size_t)n * nb + k)], f.znb[2 * ((size_t)n * nb + k) + 1]); };
      // D[e][n] = sum_k X[e][k] B[n][k],  X = [Re i (16) | Im i (16)],  D = [Re du (16) | Im du (16)]
      std::vector<double> b1((size_t)32 * 32, 0.0), b2((size_t)n2 * 32, 0.0);
      for (int k = 0; k < nb; ++k)
        for (int j = 0; j < nb; ++j) {
          const double2 z = Z(k, j);
          b1[(size_t)k * 32 + j] = -z.x;            // Re du_k -= Zr Re i_j
          b1[(size_t)k * 32 + NB + j] = z.y;        //           + Zi Im i_j
          b1[(size_t)(NB + k) * 32 + j] = -z.y;     // Im du_k -= Zi Re i_j
          b1[(size_t)(NB + k) * 32 + NB + j] = -z.x;  //         - Zr Im i_j
        }
      for (int n = 0; n < nn; ++n)                  // rows interleaved: 2n = Re dv_n, 2n+1 = Im dv_n
        for (int k = 0; k < nb; ++k) {
          const double2 z = ZN(n, k);
          b2[(size_t)(2 * n) * 32 + k] = -z.x;
          b2[(size_t)(2 * n) * 32 + NB + k] = z.y;
          b2[(size_t)(2 * n + 1) * 32 + k] = -z.y;
          b2[(size_t)(2 * n + 1) * 32 + NB + k] = -z.x;
        }
      std::vector<unsigned char> blob;
      auto put = [&blob](const void* src, size_t bytes) {
        const size_t off = (blob.size() + 127) / 128 * 128;
        blob.resize(off + bytes, 0);
        memcpy(blob.data() + off, src, bytes);
        return (int)off;
      };
      std::vector<unsigned char> i1 = image(32, b1), i2 = image(n2, b2);
      put(i1.data(), i1.size());
      env->tc_off_b2 = put(i2.data(), i2.size());
      std::vector<float> u0f(2 * NB, 0.f), wf(2 * nnp8, 0.f), vlf(NB, 0.95f), vhf(NB, 1.05f);
      std::vector<double> shd(NB, 0.0);
      std::vector<int32_t> bl16(NB, 0), bm16(NB, 1), slot(env->A), node(env->A);
      for (int k = 0; k < NB; ++k) { u0f[2 * k] = 1.f; }
      for (int k = 0; k < nb; ++k) {
        u0f[2 * k] = (float)f.u0[2 * k]; u0f[2 * k + 1] = (float)f.u0[2 * k + 1];
        vlf[k] = (float)f.vminpu[k]; vhf[k] = (float)f.vmaxpu[k]; shd[k] = f.branch_share[k];
        bl16[k] = f.branch_load[k]; bm16[k] = f.branch_model[k];
      }
      for (int n = 0; n < nn; ++n) { wf[2 * n] = (float)f.w[2 * n]; wf[2 * n + 1] = (float)f.w[2 * n + 1]; }
      for (int a = 0; a < env->A; ++a) { slot[a] = spec->agents[a].load_slot; node[a] = spec->agents[a].bus_node; }
      env->tc_off_u0 = put(u0f.data(), u0f.size() * 4);
      env->tc_off_w = put(wf.data(), wf.size() * 4);
      env->tc_off_share = put(shd.data(), shd.size() * 8);
      env->tc_off_vlo = put(vlf.data(), vlf.size() * 4);
      env->tc_off_vhi = put(vhf.data(), vhf.size() * 4);
      env->tc_off_bload = put(bl16.data(), bl16.size() * 4);
      env->tc_off_bmodel = put(bm16.data(), bm16.size() * 4);
      env->tc_off_slot = put(slot.data(), slot.size() * 4);
      env->tc_off_node = put(node.data(), node.size() * 4);
      blob.resize((blob.size() + 127) / 128 * 128, 0);
      env->tc_blob_bytes = (int)blob.size();
      env->tc_n2 = n2; env->tc_nnp8 = nnp8;
      PGW_TRY(upload(&env->tc_blob, blob.data(), blob.size())); env->own(env->tc_blob);
    }
    if (pgw::tc2_padded_chunks((nb + 7) / 8) > 0) {
      // Operand images of the FP16 tcgen05 kernel (powerflow_tc2.cu), byte-exact as they sit in
      // shared memory: canonical K-major no-swizzle UMMA tiles, element (row, k) of an image
      // with K columns at  (row/8)*SBO + (k/8)*128 + (row%8)*16 + (k%8)*2,  SBO = (K/8)*128.
      // Row / column order: 16c + j = Re (j < 8) or Im (j >= 8) of item 8c + (j % 8).
      pgw::Tc2Params& t = env->tc2;
      const int nch = pgw::tc2_padded_chunks((nb + 7) / 8), N = 16 * nch, NBP = 8 * nch;
      const size_t sbo = (size_t)(N / 8) * 128, part = (size_t)(N / 8) * sbo;
      auto pos = [](int item, bool im) { return 16 * (item / 8) + (item % 8) + (im ? 8 : 0); };
      auto Z = [&](int k, int j) { return make_double2(f.zbb[2 * ((size_t)k * nb + j)], f.zbb[2 * ((size_t)k * nb + j) + 1]); };
      auto ZN = [&](int n, int k) { return make_double2(f.znb[2 * ((size_t)n * nb + k)], f.znb[2 * ((size_t)n * nb + k) + 1]); };
      // Nodes whose voltage IS a load-branch voltage up to a real factor c (a wye load between
      // the node and ground: row n of Znb = c x row k of Zbb and w[n] = c u0[k], c = the ratio
      // of the two voltage bases) need no expansion: |v_n| = c |u_k|.
      std::vector<int32_t> dnode(NBP, -1), xnode;
      std::vector<float> dscale(NBP, 0.f);
      std::vector<double> dscale64(NBP, 0.0);
      {
        std::vector<char> taken(nb, 0);
        for (int n = 0; n < nn; ++n) {
          int hit = -1;
          double cr = 0.0;
          for (int k = 0; k < nb && hit < 0; ++k) {
            if (taken[k]) continue;
            const double ur = f.u0[2 * k], ui = f.u0[2 * k + 1], wr = f.w[2 * n], wi = f.w[2 * n + 1];
            const double den = ur * ur + ui * ui;
            if (den <= 0.0) continue;
            const double c = (wr * ur + wi * ui) / den;
            if (!(c > 0.0)) continue;
            double err = std::hypot(wr - c * ur, wi - c * ui), ref = std::hypot(wr, wi);
            for (int j = 0; j < nb; ++j) {
              const double2 a = ZN(n, j), b = Z(k, j);
              err = std::fmax(err, std::hypot(a.x - c * b.x, a.y - c * b.y));
              ref = std::fmax(ref, std::hypot(a.x, a.y));
            }
            if (err <= 1e-10 * ref) { hit = k; cr = c; }
          }
          if (hit >= 0) { taken[hit] = 1; dnode[hit] = n; dscale[hit] = (float)cr; dscale64[hit] = cr; }
          else xnode.push_back(n);
        }
      }
      const int nx = (int)xnode.size(), ncc = (nx + NBP - 1) / NBP;
      xnode.resize((size_t)std::max(ncc, 1) * NBP, -1);
      // real-ified operator rows:  D[pos(out)] = sum_k X[pos(k)] * M[pos(out)][pos(k)]
      auto realify = [&](int rows_items, int item0, int nitems, auto&& zget) {
        std::vector<double> m((size_t)N * N, 0.0);
        for (int r = 0; r < rows_items; ++r) {
          const int item = item0 + r;
          if (item >= nitems) break;
          for (int k = 0; k < nb; ++k) {
            const double2 z = zget(item, k);
            m[(size_t)pos(r, false) * N + pos(k, false)] = -z.x;   // Re out -= Zr Re i
            m[(size_t)pos(r, false) * N + pos(k, true)] = z.y;     //         + Zi Im i
            m[(size_t)pos(r, true) * N + pos(k, false)] = -z.y;    // Im out -= Zi Re i
            m[(size_t)pos(r, true) * N + pos(k, true)] = -z.x;     //         - Zr Im i
          }
        }
        return m;
      };
      auto scale_for = [](double mx) {
        return mx > 0.0 ? std::ldexp(1.0, (int)std::floor(std::log2(16384.0 / mx))) : 1.0;
      };
      auto images = [&](const std::vector<double>& m, double scale, unsigned char* dst) {
        for (int r = 0; r < N; ++r)
          for (int k = 0; k < N; ++k) {
            const double v = m[(size_t)r * N + k] * scale;
            const __half hi = __float2half_rn((float)v);
            const __half lo = __float2half_rn((float)(v - (double)__half2float(hi)));
            const size_t off = (size_t)(r / 8) * sbo + (size_t)(k / 8) * 128 + (r % 8) * 16 + (k % 8) * 2;
            memcpy(dst + off, &hi, 2);
            memcpy(dst + part + off, &lo, 2);
          }
      };
      double mx1 = 0.0, mx2 = 0.0;
      for (size_t i = 0; i < 2 * (size_t)nb * nb; ++i) mx1 = std::fmax(mx1, std::fabs(f.zbb[i]));
      for (size_t i = 0; i < 2 * (size_t)nn * nb; ++i) mx2 = std::fmax(mx2, std::fabs(f.znb[i]));
      const double sb1 = scale_for(mx1), sb2 = scale_for(mx2), xs = 2048.0;
      std::vector<unsigned char> blob((size_t)(1 + ncc) * 2 * part, 0);
      images(realify(NBP, 0, nb, Z), sb1, blob.data());
      for (int cc = 0; cc < ncc; ++cc)
        images(realify(NBP, cc * NBP, nx, [&](int slot, int k) { return ZN(xnode[slot], k); }), sb2,
               blob.data() + (size_t)(1 + cc) * 2 * part);
      t.nch = nch; t.ncc = ncc; t.nx = nx; t.part_bytes = (int)part; t.off_zn = (int)(2 * part);
      t.off_tab = (int)blob.size();
      t.xscale = (float)xs; t.descale1 = (float)(1.0 / (sb1 * xs)); t.descale2 = (float)(1.0 / (sb2 * xs));
      t.tol = (float)(f.tol > 1e-7 ? f.tol : 1e-7);
      // small feeders keep every Znb chunk resident (64 kB of images, accumulators 2 + cc)
      t.resident = ((2 + ncc) * N <= 512 && (size_t)ncc * 2 * part <= 64 * 1024) ? 1 : 0;
      t.tmem_cols = 32;
      while (t.tmem_cols < (t.resident ? 2 + ncc : 2) * N) t.tmem_cols *= 2;
      // cst = {Re u0, Im u0, vlo^2, vhi^2}, gh = (1, 0) -> 1/clamp(|u|^2), (0, 1) -> 1/|u| (model 5)
      std::vector<float> cst(4 * (size_t)NBP, 1.f), gh(2 * (size_t)NBP, 0.f), shf(NBP, 0.f), wf(2 * xnode.size(), 0.f);
      std::vector<int32_t> blp(NBP, 0), bag(NBP, -1), lptr(f.nl + 1, 0), lidx(env->A, 0), node(env->A);
      for (int k = 0; k < NBP; ++k) { cst[4 * k + 1] = 0.f; gh[2 * k] = 1.f; }
      for (int k = 0; k < nb; ++k) {
        cst[4 * k] = (float)f.u0[2 * k]; cst[4 * k + 1] = (float)f.u0[2 * k + 1];
        if (f.branch_model[k] == 5) {
          cst[4 * k + 2] = 1e-30f; cst[4 * k + 3] = 3e38f; gh[2 * k] = 0.f; gh[2 * k + 1] = 1.f;
          t.any_m5 = 1;
        } else if (f.branch_model[k] != 2) {
          cst[4 * k + 2] = (float)(f.vminpu[k] * f.vminpu[k]);
          cst[4 * k + 3] = (float)(f.vmaxpu[k] * f.vmaxpu[k]);
        }
        shf[k] = (float)(f.branch_share[k] * 1e-3);
        blp[k] = f.branch_load[k];
      }
      for (int sidx = 0; sidx < nx; ++sidx) {
        wf[2 * sidx] = (float)f.w[2 * xnode[sidx]]; wf[2 * sidx + 1] = (float)f.w[2 * xnode[sidx] + 1];
      }
      for (int a = 0; a < env->A; ++a) {
        node[a] = spec->agents[a].bus_node;
        if (spec->agents[a].load_slot >= 0) ++lptr[spec->agents[a].load_slot + 1];
      }
      for (int l = 0; l < f.nl; ++l) lptr[l + 1] += lptr[l];
      {
        std::vector<int32_t> fill(lptr.begin(), lptr.end() - 1);
        for (int a = 0; a < env->A; ++a)              // agent order inside a load slot
          if (spec->agents[a].load_slot >= 0) lidx[fill[spec->agents[a].load_slot]++] = a;
      }
      auto put = [&blob, &t](const void* src, size_t bytes) {
        const size_t off = (blob.size() + 15) / 16 * 16;
        blob.resize(off + bytes, 0);
        if (bytes) memcpy(blob.data() + off, src, bytes);
        return (int)(off - (size_t)t.off_tab);
      };
      for (int k = 0; k < nb; ++k) {                  // the one agent on the branch's load, or -2
        const int l = blp[k], cnt = lptr[l + 1] - lptr[l];
        bag[k] = cnt == 0 ? -1 : (cnt == 1 ? lidx[lptr[l]] : -2);
      }
      for (int q = 0; q < NBP / 2; ++q) {            // pairs of branches (2q, 2q + 1)
        const int k0 = 2 * q, k1 = 2 * q + 1;
        env->tc2c.pa[q] = make_float4(cst[4 * k0], cst[4 * k1], cst[4 * k0 + 1], cst[4 * k1 + 1]);
        env->tc2c.pb[q] = make_float4(cst[4 * k0 + 2], cst[4 * k1 + 2], cst[4 * k0 + 3], cst[4 * k1 + 3]);
        env->tc2c.pc[q] = make_float4(gh[2 * k0], gh[2 * k1], gh[2 * k0 + 1], gh[2 * k1 + 1]);
      }
      t.consts = &env->tc2c;
      t.t_share = put(shf.data(), shf.size() * 4);
      t.t_bload = put(blp.data(), blp.size() * 4);
      t.t_bagent = put(bag.data(), bag.size() * 4);
      t.t_w = put(wf.data(), wf.size() * 4);
      t.t_xnode = put(xnode.data(), xnode.size() * 4);
      t.t_dnode = put(dnode.data(), dnode.size() * 4);
      t.t_dscale = put(dscale.data(), dscale.size() * 4);
      // FP64 polish (powerflow_tc2.cu): one full float64 sweep + one over the rows the rewards
      // and the agents read, on by default where the rewards read the fresh voltages
      t.polish_ok = nch == 2 ? 1 : 0;
      t.polish = (t.polish_ok && env->punit != 0.0) ? 1 : 0;
      t.tol = tc2_default_tol(f.tol, t.polish);
      t.polish_row = -1;
      if (t.polish_ok) {
        pgw::Tc2Polish& kp = env->tc2p;
        for (int j = 0; j < 16; ++j)
          for (int k = 0; k < 16; ++k)
          {
            kp.zT[j * 16 + k] = (j < nb && k < nb) ? Z(k, j) : make_double2(0.0, 0.0);
            kp.z32[j * 16 + k] = make_float2((float)(kp.zT[j * 16 + k].x / xs), (float)(kp.zT[j * 16 + k].y / xs));
          }
        for (int k = 0; k < 16; ++k) {
          const bool real = k < nb;
          kp.u0[k] = real ? make_double2(f.u0[2 * k], f.u0[2 * k + 1]) : make_double2(1.0, 0.0);
          kp.share[k] = real ? f.branch_share[k] * 1e-3 : 0.0;
          kp.model[k] = real ? f.branch_model[k] : 1;
          const bool z = real && f.branch_model[k] == 2;
          kp.vlo2[k] = z ? 1.0 : (real ? f.vminpu[k] * f.vminpu[k] : 0.9025);
          kp.vhi2[k] = z ? 1.0 : (real ? f.vmaxpu[k] * f.vmaxpu[k] : 1.1025);
          kp.dscale[k] = real ? dscale64[k] : 0.0;
        }
        kp.rows = 0u;
        auto mark = [&](int node) {
          for (int k = 0; k < nb; ++k)
            if (node >= 0 && dnode[k] == node) { kp.rows |= 1u << k; return true; }
          return false;
        };
        for (int a = 0; a < env->A; ++a) mark(spec->agents[a].bus_node);
        if (env->punit != 0.0 && !mark(env->penalty_node)) t.polish_row = env->penalty_node;
        t.pconsts = &env->tc2p;
      }
      t.t_lptr = put(lptr.data(), lptr.size() * 4);
      t.t_lidx = put(lidx.data(), lidx.size() * 4);
      t.t_anode = put(node.data(), node.size() * 4);
      {
        // up to two agents per branch whose bus node derives from it (vag); the others (more
        // than two on a node, or a bus that is not a wye-load node) go to the tail list
        std::vector<int32_t> vag(2 * (size_t)NBP, -1), vtail;
        for (int a = 0; a < env->A; ++a) {
          int k = -1;
          for (int q = 0; q < NBP && k < 0; ++q)
            if (dnode[q] >= 0 && node[a] == dnode[q]) k = q;
          if (k >= 0 && vag[2 * k] < 0) vag[2 * k] = a;
          else if (k >= 0 && vag[2 * k + 1] < 0) vag[2 * k + 1] = a;
          else vtail.push_back(a);
        }
        t.ntail = (int)vtail.size();
        vtail.push_back(0);
        t.t_vag = put(vag.data(), vag.size() * 4);
        t.t_vtail = put(vtail.data(), vtail.size() * 4);
      }
      blob.resize((blob.size() + 15) / 16 * 16, 0);
      t.tab_bytes = (int)(blob.size() - (size_t)t.off_tab);
      t.off_ftab = (int)blob.size(); t.ftab_bytes = 0; t.pen_slot = -1;
      if (t.polish_ok) {                               // the fused step kernel's own section
        auto putf = [&blob, &t](const void* src, size_t bytes) {
          const size_t off = (blob.size() + 15) / 16 * 16;
          blob.resize(off + bytes, 0);
          if (bytes) memcpy(blob.data() + off, src, bytes);
          return (int)(off - (size_t)t.off_ftab);
        };
        std::vector<int32_t> aslot(std::max(env->A, 1), -1);
        for (int a = 0; a < env->A; ++a)
          for (int k = 0; k < nb; ++k)
            if (node[a] >= 0 && dnode[k] == node[a]) aslot[a] = k;
        for (int k = 0; k < nb; ++k)
          if (env->punit != 0.0 && dnode[k] == env->penalty_node) t.pen_slot = k;
        t.f_kc = putf(&env->tc2c, sizeof(env->tc2c));
        t.f_kp = putf(&env->tc2p, sizeof(env->tc2p));
        t.f_aslot = putf(aslot.data(), aslot.size() * 4);
        // B fragments of the fused kernel's mma.sync.m16n8k16 products: the realified operator
        // (rows: outputs, columns: the 16 branch currents) x scale, split into FP16 hi / lo as
        // images() does, with (Re, Im) interleaved per item along N (the outputs) and K (the
        // currents): n-tile j = outputs 4j .. 4j + 3.  In the order the registers take them:
        // [n-tile][lane][k-step][hi b0, hi b1, lo b0, lo b1], two 16-byte loads a lane.
        auto mma_frags = [&](std::vector<uint16_t>& bf, int ntiles, int nitems, double scale, auto&& zget) {
          const size_t base = bf.size();
          bf.resize(base + (size_t)ntiles * 32 * 2 * 4 * 2, 0);
          for (int j = 0; j < ntiles; ++j)
            for (int lane = 0; lane < 32; ++lane) {
              const int g = lane >> 2, tq = lane & 3;
              const int r = 4 * j + g / 2;               // output item of column 8j + g
              const bool im_out = (g & 1) != 0;
              for (int s = 0; s < 2; ++s)
                for (int reg = 0; reg < 2; ++reg)
                  for (int ii = 0; ii < 2; ++ii) {       // the two halves: Re / Im of current q
                    const int q = 8 * s + tq + 4 * reg;
                    const double2 z = (r < nitems && q < nb) ? zget(r, q) : make_double2(0.0, 0.0);
                    const double v = (im_out ? (ii ? -z.x : -z.y) : (ii ? z.y : -z.x)) * scale;
                    const __half hi = __float2half_rn((float)v);
                    const __half lo = __float2half_rn((float)(v - (double)__half2float(hi)));
                    const size_t o = base + ((((size_t)j * 32 + lane) * 2 + s) * 4 + reg) * 2 + ii;
                    memcpy(&bf[o], &hi, 2);
                    memcpy(&bf[o + 4], &lo, 2);
                  }
            }
        };
        // f_xz: 4 n-tiles of the fixed point's drops (Zbb x sb1), then 4 per chunk of 16 slots of
        // the expansion's node voltages (Znb of the expansion slots x sb2)
        std::vector<uint16_t> bf;
        mma_frags(bf, 4, nb, sb1, Z);
        mma_frags(bf, 4 * ncc, nx, sb2, [&](int slot, int k) { return ZN(xnode[slot], k); });
        t.f_xz = putf(bf.data(), bf.size() * 2);
        blob.resize((blob.size() + 15) / 16 * 16, 0);
        t.ftab_bytes = (int)(blob.size() - (size_t)t.off_ftab);
      }
      pgw::PfParams probe{};
      probe.nl = f.nl; probe.tc2 = t;
      if (pgw::tc2_smem_bytes(probe) + 6 * 1024 <= 227 * 1024) {   // + the kernel's static arrays
        PGW_TRY(upload(&env->tc2_blob, blob.data(), blob.size())); env->own(env->tc2_blob);
        env->tc2.blob = env->tc2_blob;
        // The fused step kernel serves feeders with <= 16 load branches, stock components on their
        // straight-line paths, tables that fit shared memory.
        bool ok = nch == 2 && !env->has_house && !env->ev_per_env && !env->need_scratch;
        for (int c = 0; c < spec->num_components && ok; ++c) {
          const pgw_component& k = spec->components[c];
          ok = k.type >= PGW_STORAGE && k.type <= PGW_BUILDING &&
               (k.type != PGW_BUILDING || (k.flags & PGW_F_BUILDING_FAST));
        }
        if (ok) {
          pgw::FusedParams P{};
          P.c.blob_bytes = env->comp_blob_bytes; P.c.dstride = env->dstride; P.c.istride = env->istride;
          P.f.tc2 = t; P.C = env->C; P.act_dim = env->act_dim;
          ok = pgw::step_fused_smem_bytes(P) + 2048 <= 200 * 1024;
        }
        env->fused_ok = ok;
      }
    }
    PGW_TRY(alloc_zero(&env->vmag, (size_t)nn * E)); env->own(env->vmag);
    PGW_TRY(alloc_zero(&env->vmin, E)); env->own(env->vmin);
    PGW_TRY(alloc_zero(&env->vmax, E)); env->own(env->vmax);
    PGW_TRY(alloc_zero(&env->vbus, A * E)); env->own(env->vbus);
    PGW_TRY(alloc_zero(&env->viol, E)); env->own(env->viol);
    PGW_TRY(alloc_zero(&env->iters, E)); env->own(env->iters);
  }
#undef PGW_TRY
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

static pgw::CompParams comp_params(pgw_env* env) {
  pgw::CompParams p{};
  p.E = env->E; p.A = env->A; p.e_lo = 0; p.e_hi = env->E; p.tickets = (unsigned int)env->num_ctas;
  p.blob = env->comp_blob; p.blob_bytes = env->comp_blob_bytes;
  p.off_comps = env->off_comps; p.off_dpar = env->off_dpar; p.off_ipar = env->off_ipar;
  p.work = env->work; p.num_ctas = env->num_ctas; p.max_cn = env->max_cn; p.max_dn = env->max_dn; p.max_in = env->max_in;
  p.dtab = env->dtab; p.itab = env->itab; p.dstride = env->dstride; p.istride = env->istride;
  p.sd = env->sd; p.si = env->si; p.rew_copy = env->rew_last;
  p.vmin = env->vmin; p.vmax = env->vmax; p.vbus = env->vbus;
  p.agent_p = env->agent_p; p.ep_ret = env->ep_ret;
  p.clock = env->d_clock; p.ticket = env->d_ticket;
  p.has_house = env->has_house;
  p.ev_per_env = env->ev_per_env ? 1 : 0;
#ifdef PGW_PHASE_TIMERS
  p.phase_clk = env->phase_clk + (size_t)4096 * 16;
#endif
  return p;
}

static pgw::PfParams pf_params(pgw_env* env) {
  pgw::PfParams p{};
  p.e_lo = 0; p.e_hi = env->E;
  p.E = env->E; p.A = env->A; p.nb = env->nb; p.nn = env->nn; p.nl = env->nl;
  p.nbp = env->nbp; p.nnp = env->nnp; p.max_iter = env->max_iter; p.tol = env->tol;
  p.blob = env->pf_blob; p.blob_bytes = env->pf_blob_bytes; p.stage_blob = env->pf_stage;
  p.off_u0 = env->off_u0; p.off_znbT = env->off_znbT; p.off_w = env->off_w;
  p.off_share = env->off_share; p.off_vmin = env->off_vmin; p.off_vmax = env->off_vmax;
  p.off_bload = env->off_bload; p.off_bmodel = env->off_bmodel; p.off_slot = env->off_slot;
  p.off_node = env->off_node; p.u_state = env->u_state; p.rew_copy = env->rew_last;
  p.tc_blob = env->tc_blob; p.tc_blob_bytes = env->tc_blob_bytes; p.tc_n2 = env->tc_n2;
  p.tc_nnp8 = env->tc_nnp8; p.tc_off_b2 = env->tc_off_b2; p.tc_off_u0 = env->tc_off_u0;
  p.tc_off_w = env->tc_off_w; p.tc_off_share = env->tc_off_share; p.tc_off_vlo = env->tc_off_vlo;
  p.tc_off_vhi = env->tc_off_vhi; p.tc_off_bload = env->tc_off_bload;
  p.tc_off_bmodel = env->tc_off_bmodel; p.tc_off_slot = env->tc_off_slot;
  p.tc_off_node = env->tc_off_node;
  p.tc_tol = (float)(env->tol > 1e-7 ? env->tol : 1e-7);
  p.tc2 = env->tc2;
  p.dtab = env->dtab; p.dstride = env->dstride;
  p.vmag = env->vmag; p.vmin = env->vmin; p.vmax = env->vmax; p.vbus = env->vbus;
  p.iters = env->iters; p.ep_ret = env->ep_ret; p.viol = env->viol;
  p.penalty_node = env->penalty_node; p.pvlo = env->pvlo; p.pvhi = env->pvhi; p.punit = env->punit;
  p.clock = env->d_clock; p.ticket = env->d_ticket;
#ifdef PGW_PHASE_TIMERS
  p.phase_clk = env->phase_clk;
#endif
  return p;
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
  return env->max_cn * (int)sizeof(pgw_component) + env->max_dn * 8 + env->max_in * 4 +
         env->dstride * 8 + env->istride * 4 +
         ((reset ? env->need_scratch_reset : env->need_scratch) ? 35 * 64 * 8 : 0);
}

// io32: obs is a float array (pgw_reset_f32), else double
static int reset_impl(pgw_env* env, const double* init_soc, void* obs, bool io32, void* cuda_stream) {
  if (!env || !obs) return fail(PGW_ERR_INVALID, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  PGW_CUDA(cudaMemsetAsync(env->d_clock, 0, sizeof(int), s));
  PGW_CUDA(cudaMemsetAsync(env->d_ticket, 0, sizeof(unsigned int), s));
  if (env->has_feeder) {
    pgw::PfParams pf = pf_params(env);
    pf.event_mode = 0; pf.advance_clock = 0; pf.agent_p = nullptr; pf.rew = nullptr;
    pf.punit = 0.0; pf.warm_start = 0;
    PGW_CUDA(launch_pf(env, pf, s));
    ++env->launches;
  }
  pgw::CompParams cp = comp_params(env);
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
  pgw::CompParams cp = comp_params(env);
  const bool hook = env->has_feeder && env->punit != 0.0;   // power flow finishes the rewards
  cp.event_mode = 1; cp.advance_clock = env->has_feeder ? 0 : 1; cp.owns_reward = hook ? 0 : 1;
  cp.actions = actions; cp.obs = obs; cp.rew = rew; cp.done = done; cp.io32 = io32 ? 1 : 0;
  cp.pdl_trigger = pdl_trigger;
  cp.e_lo = e_lo; cp.e_hi = e_hi; cp.tickets = (unsigned int)(env->num_ctas * chunks);
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
  pgw::PfParams pf = pf_params(const_cast<pgw_env*>(env));
  pf.event_mode = 1; pf.reward_hook = (env->punit != 0.0) ? 1 : 0;
  if (pgw::tc2_smem_bytes(pf) > 112 * 1024) return 0;   // two power-flow CTAs + component CTAs per SM
  return env->num_ctas <= 148 * 4 ? 1 : 2;
}

static pgw::PfParams step_pf_params(pgw_env* env, double* rew, int e_lo, int e_hi, unsigned int tickets,
                                    bool pdl) {
  pgw::PfParams pf = pf_params(env);
  pf.event_mode = 1; pf.advance_clock = 1; pf.agent_p = env->agent_p; pf.rew = rew;
  pf.reward_hook = (env->punit != 0.0) ? 1 : 0;
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
      pgw::PfParams pf = pf_params(env);
      pf.event_mode = 1; pf.reward_hook = (env->punit != 0.0) ? 1 : 0;
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
    case PGW_FIELD_VOLTAGES: *ptr = env->vmag; *want = (size_t)env->nn * E * 8; break;
    case PGW_FIELD_VMIN: *ptr = env->vmin; *want = E * 8; break;
    case PGW_FIELD_VMAX: *ptr = env->vmax; *want = E * 8; break;
    case PGW_FIELD_VBUS: *ptr = env->vbus; *want = A * E * 8; break;
    case PGW_FIELD_PF_ITERS: *ptr = env->iters; *want = E * 4; break;
    case PGW_FIELD_EP_RETURN: *ptr = env->ep_ret; *want = A * E * 8; break;
    case PGW_FIELD_PF_STATE: *ptr = env->u_state; *want = (size_t)env->nbp * E * 16; break;
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
      PGW_CUDA(cudaMemcpyAsync(env->comp_blob + env->off_dpar, dpar, (size_t)dpar_len * sizeof(double),
                               cudaMemcpyHostToDevice, s));
  }
  if (dtab)
    PGW_CUDA(cudaMemcpyAsync(env->dtab, dtab, (size_t)env->num_events * env->dstride * sizeof(double),
                             cudaMemcpyHostToDevice, s));
  if (itab && env->istride)
    PGW_CUDA(cudaMemcpyAsync(env->itab, itab, (size_t)env->num_events * env->istride * sizeof(int32_t),
                             cudaMemcpyHostToDevice, s));
  PGW_CUDA(cudaStreamSynchronize(s));
  return PGW_OK;
}

int pgw_pf_solve(pgw_env* env, const double* load_kw, const double* load_kvar,
                 void* cuda_stream) {
  if (!env || !load_kw || !load_kvar) return fail(PGW_ERR_INVALID, "null argument");
  if (!env->has_feeder) return fail(PGW_ERR_INVALID, "this env has no feeder");
  pgw::PfParams pf = pf_params(env);
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
  p.E = env->E; p.A = env->A; p.nn = env->nn;
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
int pgw_debug_num_comp_ctas(pgw_env* env) { return env ? env->num_ctas : 0; }
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
      if (value == 2 && !env->tc2_blob)
        return fail(PGW_ERR_INVALID, "FP16 tensor-core power flow needs a feeder with <= 88 load "
                                     "branches whose tables fit shared memory");
      if (value == 1 && !env->tc_blob)
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
      if (value > 0 && !env->tc2.polish_ok)
        return fail(PGW_ERR_INVALID, "the FP64 polish serves feeders with <= 16 load branches");
      env->tc2.polish = value;
      if (!env->tc2_tol_set) env->tc2.tol = tc2_default_tol(env->tol, value);
      break;
    case PGW_OPT_PF_TC_TOL_NANO:
      if (value < 10 || value > 100000) return fail(PGW_ERR_INVALID, "tolerance out of range (1e-8..1e-4)");
      env->tc2.tol = (float)(value * 1e-9);
      env->tc2_tol_set = true;
      break;
    default: return fail(PGW_ERR_INVALID, "unknown option");
  }
  // the captured graphs bake the options in
  env->drop_graphs();
  return PGW_OK;
}

}  // extern "C"
