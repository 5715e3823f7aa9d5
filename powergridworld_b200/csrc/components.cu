// K1-K5 + the lagged part of K7, fused: one thread per (env, agent) steps all of the
// agent's components in order, writes the agent's observation rows, its real power
// (the input of the power flow) and its reward.  Streams structure-of-arrays state
// (env index fastest => fully coalesced 8-byte accesses).
//
// Everything that is shared by all envs -- the static tables (agents, component
// descriptors, parameters) and the event row of this step (PV profile value, building
// weather row, EV window lists, base feeder load, done flag) -- is staged once per CTA
// into shared memory with two TMA bulk copies (cp.async.bulk -> UBLKCP) and read from
// there as warp-uniform broadcasts, so the only global traffic of a thread is its own
// per-env state, actions and outputs.
//
// Replaces HOT LOOP 1-3 of gridworld/multiagent_env.py:165-181 and gridworld/base.py:125-137.
// Compiled with -fmad=false (see component_math.cuh).
#include <type_traits>

#include "component_math.cuh"
#include "internal.cuh"
#include "tma.cuh"

namespace pgw {

// HOUSE: the scenario contains Home-Steward houses (their code stays out of the other kernel);
// TEL: some of their components record step_meta telemetry.
// EVENV: some charging station runs on per-env rosters (PGW_F_EV_PER_ENV).
// IO32: the caller's actions and observations are float arrays (p.io32), else double.
template <bool HOUSE, bool TEL, bool EVENV = false, bool IO32 = false>
__global__ void __launch_bounds__(64, 10) component_kernel(const CompParams p) {
  using IoT = typename std::conditional<IO32, float, double>::type;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t mbar[2];
  // [comps slice | dpar slice | ipar slice | double event row | int event row | scratch]
  const size_t b_comps = (size_t)p.max_cn * sizeof(pgw_component);
  const size_t b_dpar = (size_t)p.max_dn * 8, b_ipar = (size_t)p.max_in * 4;
  pgw_component* s_comps = reinterpret_cast<pgw_component*>(smem_raw);
  double* s_dpar = reinterpret_cast<double*>(smem_raw + b_comps);
  int32_t* s_ipar = reinterpret_cast<int32_t*>(smem_raw + b_comps + b_dpar);
  const size_t static_bytes = b_comps + b_dpar + b_ipar;
  double* drow = reinterpret_cast<double*>(smem_raw + static_bytes);
  int32_t* irow = reinterpret_cast<int32_t*>(smem_raw + static_bytes + (size_t)p.dstride * 8);
  double* scratch = reinterpret_cast<double*>(
      smem_raw + static_bytes + (size_t)p.dstride * 8 + (size_t)p.istride * 4);

  // the three independent global reads of the prologue, issued back to back
  const CtaWork wk = p.work[blockIdx.x];
  const int a = wk.agent;
  const AgentSlice sl = wk.sl;
  const pgw_agent ag = reinterpret_cast<const pgw_agent*>(p.blob)[a];
#ifdef PGW_PHASE_TIMERS
#define C_STAMP(k)                                                                        \
  do {                                                                                    \
    if (p.phase_clk != nullptr && threadIdx.x == 0) p.phase_clk[(size_t)blockIdx.x * 8 + (k)] = clock64(); \
  } while (0)
  if (p.phase_clk != nullptr && threadIdx.x == 0) p.phase_clk[(size_t)blockIdx.x * 8] = (long long)global_timer_ns();
#else
#define C_STAMP(k) do { } while (0)
#endif
  C_STAMP(2);
  const int clk = p.event_mode == 0 ? -1 : *p.clock;
  unsigned int my_ticket = 0u;                        // thread 0, when this kernel advances the clock
  const int ev = clk + 1;
  // Two staging phases so that the latency of reading the device clock (which selects the
  // event row) overlaps the copy of the static tables and the threads' own prefetches.
  // A CTA serves one agent, so only that agent's slice of the tables is staged.
  if (threadIdx.x == 0) {
    mbar_init(&mbar[0], 1);
    mbar_init(&mbar[1], 1);
    const uint32_t cb = (uint32_t)sl.c_n * (uint32_t)sizeof(pgw_component);
    const uint32_t db = (uint32_t)sl.d_n * 8u, ib = (uint32_t)sl.i_n * 4u;
    mbar_expect_tx(&mbar[0], cb + db + ib);
    tma_bulk_g2s(s_comps, p.blob + p.off_comps + (size_t)sl.c_lo * sizeof(pgw_component), cb, &mbar[0]);
    if (db) tma_bulk_g2s(s_dpar, p.blob + p.off_dpar + (size_t)sl.d_lo * 8, db, &mbar[0]);
    if (ib) tma_bulk_g2s(s_ipar, p.blob + p.off_ipar + (size_t)sl.i_lo * 4, ib, &mbar[0]);
    const uint32_t dbytes = (uint32_t)p.dstride * 8u, ibytes = (uint32_t)p.istride * 4u;
    mbar_expect_tx(&mbar[1], dbytes + ibytes);
    tma_bulk_g2s(drow, p.dtab + (size_t)ev * p.dstride, dbytes, &mbar[1]);
    if (ibytes) tma_bulk_g2s(irow, p.itab + (size_t)ev * p.istride, ibytes, &mbar[1]);
    if (p.advance_clock) my_ticket = clock_take_ticket(p.ticket, clk);
  }
  // Programmatic dependent launch of the power-flow kernel (pdl_trigger 1): its CTAs may start
  // their prologue (tables, TMEM, prefetches) now and block in griddepcontrol.wait until this
  // grid has completed.  They advance the clock, hence only after this whole CTA has read it:
  // the barrier's predicate makes it wait for every thread's clock value.
  if (p.pdl_trigger == 1) {
    if (!__syncthreads_or(ev < 0)) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  } else {
    __syncthreads();
  }
  C_STAMP(3);
  mbar_wait(&mbar[0], 0);
  C_STAMP(4);

  const int event = ev;
  const pgw_component* comps = s_comps - sl.c_lo;      // indexed by absolute component number

  AgentIOT<IoT, IoT> io;
  io.scr.p = scratch + threadIdx.x;          // [kScratchDoubles][blockDim.x]: conflict-free
  io.scr.stride = blockDim.x;
  io.E = p.E;
  io.actions = static_cast<const IoT*>(p.actions);
  io.aE = p.E;
  io.ae0 = 0;
  io.obs = static_cast<IoT*>(p.obs);
  io.sd = p.sd;
  io.si = p.si;
  io.init_soc = p.init_soc;
  io.clip_init_soc = p.clip_init_soc;
  io.vmin = p.vmin;
  io.vmax = p.vmax;
  io.vbus = p.vbus;
  io.dpar = s_dpar - sl.d_lo;                          // absolute dpar / ipar offsets
  io.ipar = s_ipar - sl.i_lo;
  io.drow = drow;
  io.irow = irow;

  // Persistent CTA: the tables are staged once, then the CTA walks env blocks of its agent.
  bool first = true;
  for (int e = p.e_lo + wk.j * blockDim.x + threadIdx.x; e - (int)threadIdx.x < p.e_hi;
       e += wk.n * blockDim.x) {
    if (e < p.e_hi && p.event_mode != 0) {
      // pull this thread's action and (small) state rows towards the SM early
      for (int ci = ag.comp_begin; ci < ag.comp_end; ++ci) {
        const pgw_component c = comps[ci];
        const int na = c.type == PGW_BUILDING ? 6 : 1;
        for (int r = 0; r < na; ++r)
          asm volatile("prefetch.global.L1 [%0];"
                       ::"l"(static_cast<const IoT*>(p.actions) + (size_t)(c.act_off + r) * p.E + e));
        const int ns = c.type == PGW_BUILDING ? 6 : (c.type == PGW_STORAGE ? 1 : 0);
        for (int r = 0; r < ns; ++r)
          asm volatile("prefetch.global.L1 [%0];" ::"l"(p.sd + (size_t)(c.sd_off + r) * p.E + e));
      }
    }
    if (first) {
      mbar_wait(&mbar[1], 0);                  // event row has landed
      first = false;
      C_STAMP(5);
    }
    if (e < p.e_hi) {
      const size_t ae = (size_t)a * p.E + e;
      if (p.event_mode == 0) {
        if (HOUSE && is_house(ag, comps)) house_reset<TEL>(ag, comps, io, e, p.first_reset != 0);
        else agent_reset<EVENV>(ag, comps, io, e);
        p.agent_p[ae] = 0.0;
        p.ep_ret[ae] = 0.0;
      } else {
        double pw, rw, er = 0.0;
        if (p.owns_reward)                      // issued early: its latency hides behind the step
          asm volatile("ld.global.f64 %0, [%1];" : "=d"(er) : "l"(p.ep_ret + ae));
        if (HOUSE && is_house(ag, comps)) house_step<TEL>(ag, comps, io, e, pw, rw);
        else agent_step<EVENV>(ag, comps, io, e, pw, rw);
        p.agent_p[ae] = pw;
        p.rew[ae] = rw;
        if (p.owns_reward) {                    // no feeder / no penalty hook: the reward is final
          p.ep_ret[ae] = er + rw;
          p.rew_copy[ae] = rw;
        }
        if (a == 0) p.done[e] = drow[0] != 0.0 ? 1 : 0;
      }
    }
  }
  // A CTA whose first block lies outside [e_lo, e_hi) (a chunk of the staged host step with fewer
  // blocks than the agent has CTAs) never entered the loop: the event-row copy may still be
  // writing this CTA's shared memory, so it must land before the CTA exits.
  if (first) mbar_wait(&mbar[1], 0);
  C_STAMP(6);
  if (p.pdl_trigger == 2) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (p.advance_clock && threadIdx.x == 0)
    clock_advance_if_last(my_ticket, p.ticket, p.clock, clk, p.tickets);
#ifdef PGW_PHASE_TIMERS
  if (p.phase_clk != nullptr && threadIdx.x == 0) p.phase_clk[(size_t)blockIdx.x * 8 + 1] = (long long)global_timer_ns();
#endif
}

template <bool IO32>
static bool is_component_kernel_io(const void* func) {
  return func == (const void*)component_kernel<false, false, false, IO32> ||
         func == (const void*)component_kernel<true, false, false, IO32> ||
         func == (const void*)component_kernel<true, true, false, IO32> ||
         func == (const void*)component_kernel<false, false, true, IO32> ||
         func == (const void*)component_kernel<true, false, true, IO32> ||
         func == (const void*)component_kernel<true, true, true, IO32>;
}

bool is_component_kernel(const void* func) {
  return is_component_kernel_io<false>(func) || is_component_kernel_io<true>(func);
}

template <bool IO32>
static auto component_kernel_for(const CompParams& p) {
  if (p.ev_per_env)
    return p.has_house ? (p.has_house > 1 ? component_kernel<true, true, true, IO32>
                                          : component_kernel<true, false, true, IO32>)
                       : component_kernel<false, false, true, IO32>;
  return p.has_house ? (p.has_house > 1 ? component_kernel<true, true, false, IO32>
                                        : component_kernel<true, false, false, IO32>)
                     : component_kernel<false, false, false, IO32>;
}

cudaError_t launch_components(const CompParams& p, int smem_bytes, cudaStream_t s) {
  const int threads = 64;      // small CTAs: a 4096-env batch still reaches every SM
  dim3 grid(p.num_ctas);       // the CTA -> (agent, env blocks) table is built in pgw_create
  auto kern = p.io32 ? component_kernel_for<true>(p) : component_kernel_for<false>(p);
  if (smem_bytes > 48 * 1024) {
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
    if (err != cudaSuccess) return err;
  }
  kern<<<grid, threads, smem_bytes, s>>>(p);
  return cudaGetLastError();
}

}  // namespace pgw
