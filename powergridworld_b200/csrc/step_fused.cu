// The whole step of an IEEE-13 class scenario in ONE kernel (replaces HOT LOOP 1-3 of
// gridworld/multiagent_env.py:165-189 + the OpenDSS solve of distribution_system/opendss.py:134
// + the reward hook of examples/marl/openai/train.py:51-88 for a tile of envs):
//
//   component steps  ->  nominal power of the load branches  ->  float32 fixed point
//   ->  float64 polish  ->  node-voltage expansion  ->  bus voltages, penalty, rewards
//
// A CTA of 512 threads owns a tile of 32 envs end to end.  Thread (w, e): warp w, lane e = env
// row of the tile -- every warp sees all 32 envs of the tile on its lanes, so everything that is
// per env but spread over warps (16 load branches, up to 16 components in flight) is warp
// uniform in control flow and coalesced (32 consecutive doubles of a state row) in memory.
//
// * Components: warp w steps the components w, w + 16, ... of the scenario (a component of a
//   MultiComponentEnv does not see its siblings, gridworld/base.py:125-137), writes their
//   observations and state, and leaves real power and reward in shared memory; the agents'
//   sums (in component order, as the reference adds them) stay on chip -- no agent_p / reward
//   round trip through HBM, no second launch, one clock read, one staging of the event row.
// * Power flow: warp w owns load branch w.  One iteration of u <- u0 - Zbb i(u) is: the current
//   of my branch into a [k][env] float2 array (conflict free, double-buffered by iteration
//   parity), one CTA barrier, then the new drop of my branch from the env's nb currents against
//   the Zbb row (Zbb^T / xscale in shared memory, warp-uniform broadcasts), two FFMA chains on
//   the FP32 pipe.  At 32 envs per tile a tensor-core contraction buys nothing: its latency was
//   the hand-offs around the MMA (DESIGN.md section 4.3d).  Per-env convergence: max |d drop|
//   over the env's 16 branch threads through a shared-memory atomicMax; converged envs freeze
//   their currents (their drop reproduces itself); every warp knows `all envs converged` from a
//   vote over its own lanes.
// * Polish: the fixed point's iteration once more with correctly rounded currents, then float64
//   sweeps u <- u0 - Zbb i(u) on the SIMT pipe, one branch per thread (the env's currents through
//   shared memory), spread over 16 warps and -- with 32-env tiles -- over every SM of the GPU:
//   ~0.4 us per sweep at 4096 envs instead of ~3 us in the 128-env tiles of powerflow_tc2.cu.
// * Expansion v = w - Znb i for the nodes that are not a wye-load node: the same float32 row
//   product against Znb^T / xscale from the fixed point's final currents, one node slot per
//   thread and chunk of 16 slots.
//
// Compiled -fmad=false like components.cu (the component arithmetic must round like NumPy);
// the power-flow code spells out its fused multiply-adds.
#include <type_traits>

#include "component_math.cuh"
#include "internal.cuh"
#include "tc2_common.cuh"
#include "tma.cuh"

namespace pgw {

constexpr int SF_ENVS = 32;                            // envs per tile = lanes of a warp
constexpr int SF_WARPS = 16;
constexpr int SF_THREADS = SF_ENVS * SF_WARPS;

struct SfLayout {                                      // byte offsets into dynamic shared memory
  uint32_t tab, ftab, blob, drow, irow, i32, i64, dmax, part, vn, cp, cr, act, total;
};

__host__ __device__ inline SfLayout sf_layout(const FusedParams& P) {
  SfLayout L;
  uint32_t o = 0;
  auto take = [&o](uint32_t bytes) {
    const uint32_t at = o;
    o += (bytes + 127u) & ~127u;
    return at;
  };
  L.tab = take((uint32_t)P.f.tc2.tab_bytes);
  L.ftab = take((uint32_t)P.f.tc2.ftab_bytes);
  L.blob = take((uint32_t)P.c.blob_bytes);
  L.drow = take((uint32_t)P.c.dstride * 8u);
  L.irow = take((uint32_t)P.c.istride * 4u + 16u);
  L.i32 = take(2u * 16u * SF_ENVS * 8u);               // fixed-point currents, [parity][k][env] float2
  L.i64 = take(16u * SF_ENVS * 16u);                   // currents of a polish sweep
  L.dmax = take(3u * SF_ENVS * 4u);
  L.part = take(2u * 16u * SF_ENVS * 4u);              // per-branch min / max |v| partials
  L.vn = take(16u * SF_ENVS * 8u);                     // |v| of each branch's wye node (penalty, bus voltages)
  L.cp = take((uint32_t)P.C * SF_ENVS * 8u);           // component real power
  L.cr = take((uint32_t)P.C * SF_ENVS * 8u);           // component reward
  L.act = take((uint32_t)P.act_dim * SF_ENVS * 8u);    // the tile's actions, [act_dim][32]
  L.total = o;
  return L;
}

// Phase stamps of tools/phase_probe.py (instrumented build only, -DPGW_PHASE_TIMERS): thread 0 of
// every CTA records the SM clock at the phase boundaries of its first tile.
#ifdef PGW_PHASE_TIMERS
#ifdef PGW_STAMP_SECOND_TILE                           // the CTA's SECOND tile: tables, TMEM, code already there
#define SF_STAMP_TILE (!first_tile)
#else
#define SF_STAMP_TILE first_tile
#endif
#define SF_STAMP(k)                                                                  \
  do {                                                                               \
    if (pf.phase_clk != nullptr && threadIdx.x == 0 && SF_STAMP_TILE)                \
      pf.phase_clk[(size_t)(blockIdx.x + P.e_lo / SF_ENVS) * 16 + (k)] = clock64();    \
  } while (0)
#else
#define SF_STAMP(k) do { } while (0)
#endif

// IO32: the caller's actions and observations are float arrays (P.c.io32), else double.
template <bool ANY_M5, bool IO32 = false>
__global__ void __launch_bounds__(SF_THREADS, 1)
    step_fused_kernel(const __grid_constant__ FusedParams P) {
  using IoT = typename std::conditional<IO32, float, double>::type;
  extern __shared__ __align__(1024) unsigned char sf_smem[];
  __shared__ __align__(8) uint64_t mbar_tab, mbar_ev, mbar_act;
  const CompParams& pc = P.c;
  const PfParams& pf = P.f;
  const Tc2Params& t = pf.tc2;
  const SfLayout L = sf_layout(P);
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int w = __shfl_sync(0xffffffffu, tid >> 5, 0);  // provably warp uniform
  const int E = pc.E;

  unsigned char* sT = sf_smem + L.tab;
  // per-branch constants of the load model and the float64 polish tables: shared memory, every
  // read a warp-uniform broadcast (as kernel parameters they were 7 kB of cold constant-cache lines)
  const Tc2Consts& kc = *reinterpret_cast<const Tc2Consts*>(sf_smem + L.ftab + t.f_kc);
  const Tc2Polish& kp = *reinterpret_cast<const Tc2Polish*>(sf_smem + L.ftab + t.f_kp);
  const int32_t* aslot = reinterpret_cast<const int32_t*>(sf_smem + L.ftab + t.f_aslot);
  const float2* z32 = kp.z32;                          // Zbb^T / xscale
  const float2* xz = reinterpret_cast<const float2*>(sf_smem + L.ftab + t.f_xz);   // Znb^T / xscale, [k][slot]
  unsigned char* sBlob = sf_smem + L.blob;
  double* drow = reinterpret_cast<double*>(sf_smem + L.drow);
  int32_t* irow = reinterpret_cast<int32_t*>(sf_smem + L.irow);
  float2* sI32 = reinterpret_cast<float2*>(sf_smem + L.i32);       // [2][16][env]
  double2* sI64 = reinterpret_cast<double2*>(sf_smem + L.i64);
  int* sDmax = reinterpret_cast<int*>(sf_smem + L.dmax);           // [3][env] float bits
  float* sVmn = reinterpret_cast<float*>(sf_smem + L.part);        // [16][env]
  float* sVmx = sVmn + 16 * SF_ENVS;
  double* sVn = reinterpret_cast<double*>(sf_smem + L.vn);         // [16][env]
  double* sCp = reinterpret_cast<double*>(sf_smem + L.cp);         // [C][env]
  double* sCr = reinterpret_cast<double*>(sf_smem + L.cr);
  IoT* sAct = reinterpret_cast<IoT*>(sf_smem + L.act);

  // ---- prologue: clock, staging of everything that is shared by the envs
  bool first_tile = true;
#ifdef PGW_PHASE_TIMERS
  if (pf.phase_clk != nullptr && threadIdx.x == 0) pf.phase_clk[(size_t)(blockIdx.x + P.e_lo / SF_ENVS) * 16 + 12] = (long long)global_timer_ns();
#endif
  SF_STAMP(0);
  const int tiles0 = (P.e_hi - P.e_lo + SF_ENVS - 1) / SF_ENVS;
  // Pull the first tile's state rows (double state, warm-start voltages, episode returns, lagged
  // grid variables) towards L2 while the clock, the tables and the operand images are in flight:
  // eight 32-byte sectors per 256-byte row segment, rows spread over the warps.
  if ((int)blockIdx.x < tiles0 && lane < 16 && pf.warm_start && w < pf.nb) {   // 16-byte elements
    const size_t e0 = (size_t)P.e_lo + (size_t)blockIdx.x * SF_ENVS + (size_t)lane * 2;
    if (e0 < (size_t)P.e_hi) asm volatile("prefetch.global.L2 [%0];" ::"l"(pf.u_state + (size_t)w * E + e0));
  }
  if ((int)blockIdx.x < tiles0 && lane < 8) {
    const size_t e0 = (size_t)P.e_lo + (size_t)blockIdx.x * SF_ENVS + (size_t)lane * 4;
    if (e0 < (size_t)P.e_hi) {
      for (int r = w; r < P.sd_rows; r += SF_WARPS) asm volatile("prefetch.global.L2 [%0];" ::"l"(pc.sd + (size_t)r * E + e0));
      for (int a = w; a < pc.A; a += SF_WARPS) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(pf.ep_ret + (size_t)a * E + e0));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(pc.vbus + (size_t)a * E + e0));
      }
      if (w == 0) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(pc.vmin + e0));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(pc.vmax + e0));
      }
    }
  }
  // The parameter block sits in the constant bank and is cold in this SM's constant cache: one
  // lane per warp touches its 64-byte lines now, in parallel, instead of every first use of a
  // field paying its own miss later on the critical path.
  if (lane == 0) {
    constexpr int kLines = (int)((sizeof(FusedParams) + 63) / 64);
    for (int l = w; l < kLines; l += SF_WARPS) {
      const int v = reinterpret_cast<const int*>(&P)[l * 16];
      asm volatile("" ::"r"(v));
    }
  }
  const int span = P.e_hi - P.e_lo;
  const int tiles = (span + SF_ENVS - 1) / SF_ENVS;
  // The actions of a (full) tile are fetched into shared memory by TMA bulk copies, one 256-byte
  // (float: 128-byte) row segment each, issued by warp 1 at kernel entry / while the previous tile's power flow
  // runs: the component steps then find them on chip.  (The first fetch used to be issued after
  // the tables had landed: a second ~1.4 us TMA round trip in front of the component steps.)
  // With actions in HOST memory this is what decouples the PCIe reads from the component code, and
  // CTA b delays its first fetch by b x stagger_cycles so that the link serves the tiles in order
  // -- the first tiles write their observations (GPU -> host) while the last ones still wait for
  // their actions (host -> GPU).
  // (a bulk copy needs a 16-byte aligned source: every row segment of the tile must start on one.  A float32
  // caller's array may start 4 or 8 bytes past a 16-byte boundary, e.g. a view into a larger tensor: its
  // tiles then read their actions from global memory)
  constexpr int kAlign = 16 / (int)sizeof(IoT);
  const bool act_aligned = !IO32 || (reinterpret_cast<uintptr_t>(pc.actions) & 15u) == 0;
  auto tile_in_smem = [&](int tile) {
    const int e0 = P.e_lo + tile * SF_ENVS;
    return act_aligned && (E % kAlign == 0) && (e0 % kAlign == 0) && e0 + SF_ENVS <= P.e_hi;
  };
  auto fetch_actions = [&](int tile) {                 // warp 1
    if (tile < tiles && tile_in_smem(tile)) {
      const int e0 = P.e_lo + tile * SF_ENVS;
      if (lane == 0) mbar_expect_tx(&mbar_act, (uint32_t)P.act_dim * SF_ENVS * (uint32_t)sizeof(IoT));
      __syncwarp();
      for (int r = lane; r < P.act_dim; r += 32)
        tma_bulk_g2s(sAct + (size_t)r * SF_ENVS, static_cast<const IoT*>(pc.actions) + (size_t)r * E + e0,
                     SF_ENVS * (uint32_t)sizeof(IoT), &mbar_act);
    }
  };
  if (w == 1) {
    if (lane == 0) mbar_init(&mbar_act, 1);
    __syncwarp();
    if (P.stagger_cycles > 0) {
      const long long c0 = clock64(), wait = (long long)blockIdx.x * P.stagger_cycles;
      while (clock64() - c0 < wait) { }
    }
    fetch_actions(blockIdx.x);
  }
  const bool host_event = P.event >= 0;                // CTA uniform
  const int clk = host_event ? P.event - 1 : *pc.clock;
  unsigned int my_ticket = 0u;
  const int event = clk + 1;
  if (tid == 0) {
    mbar_init(&mbar_tab, 1);
    mbar_init(&mbar_ev, 1);
    mbar_expect_tx(&mbar_tab, (uint32_t)t.tab_bytes + (uint32_t)t.ftab_bytes + (uint32_t)pc.blob_bytes);
    tma_bulk_g2s(sBlob, pc.blob, (uint32_t)pc.blob_bytes, &mbar_tab);
    tma_bulk_g2s(sT, t.blob + t.off_tab, (uint32_t)t.tab_bytes, &mbar_tab);
    tma_bulk_g2s(sf_smem + L.ftab, t.blob + t.off_ftab, (uint32_t)t.ftab_bytes, &mbar_tab);
    // last: the event row's address waits for the device clock
    const uint32_t dbytes = (uint32_t)pc.dstride * 8u, ibytes = (uint32_t)pc.istride * 4u;
    mbar_expect_tx(&mbar_ev, dbytes + ibytes);
    tma_bulk_g2s(drow, pc.dtab + (size_t)event * pc.dstride, dbytes, &mbar_ev);
    if (ibytes) tma_bulk_g2s(irow, pc.itab + (size_t)event * pc.istride, ibytes, &mbar_ev);
    if (!host_event) my_ticket = clock_take_ticket(pc.ticket, clk);
  }
  __syncthreads();                                     // barriers initialised
  SF_STAMP(1);
  mbar_wait(&mbar_tab, 0);
  SF_STAMP(2);

  const pgw_agent* agents = reinterpret_cast<const pgw_agent*>(sBlob);
  const pgw_component* comps = reinterpret_cast<const pgw_component*>(sBlob + pc.off_comps);
  const float* share = reinterpret_cast<const float*>(sT + t.t_share);
  const int32_t* bload = reinterpret_cast<const int32_t*>(sT + t.t_bload);
  const float2* wx = reinterpret_cast<const float2*>(sT + t.t_w);
  const int32_t* xnode = reinterpret_cast<const int32_t*>(sT + t.t_xnode);
  const int32_t* dnode = reinterpret_cast<const int32_t*>(sT + t.t_dnode);
  const float* dscale = reinterpret_cast<const float*>(sT + t.t_dscale);
  const int32_t* lptr = reinterpret_cast<const int32_t*>(sT + t.t_lptr);
  const int32_t* lidx = reinterpret_cast<const int32_t*>(sT + t.t_lidx);
  const int32_t* anode = reinterpret_cast<const int32_t*>(sT + t.t_anode);

  AgentIOT<IoT, IoT> io;
  io.scr.p = nullptr;                                  // table-driven building path: not in this kernel
  io.scr.stride = 0;
  io.E = E;
  io.actions = static_cast<const IoT*>(pc.actions);
  io.aE = E;
  io.ae0 = 0;
  io.obs = static_cast<IoT*>(pc.obs);
  io.sd = pc.sd;
  io.si = pc.si;
  io.init_soc = nullptr;
  io.clip_init_soc = 0;
  io.vmin = pc.vmin;
  io.vmax = pc.vmax;
  io.vbus = pc.vbus;
  io.dpar = reinterpret_cast<const double*>(sBlob + pc.off_dpar);
  io.ipar = reinterpret_cast<const int32_t*>(sBlob + pc.off_ipar);
  io.drow = drow;
  io.irow = irow;

  const int b = w;                                     // my load branch
  const float xs = t.xscale, ds1 = t.descale1;
  const float rds1 = 1.f / ds1;                        // a power of two: the rescaling is exact
  const float tol_s = t.tol / ds1;
  const float4 cst = t2_cst(kc, b);
  const float2 gh = ANY_M5 ? t2_gh(kc, b) : make_float2(1.f, 0.f);

  // acc - sum_k z[k zs] i_k over the nb currents of my env (cur: [k][env], scaled by xscale like
  // t2_current's; z: a column of Zbb^T or Znb^T over xscale, warp-uniform broadcasts): two FFMA
  // chains on the FP32 pipe, summed at the end.
  auto zdot = [&](float2 acc, const float2* z, int zs, const float2* cur) {
    float2 a1 = make_float2(0.f, 0.f);
#pragma unroll 2
    for (int jj = 0; jj + 1 < pf.nb; jj += 2) {
      t2_cmac_sub32(acc, z[jj * zs], cur[jj * SF_ENVS + lane]);
      t2_cmac_sub32(a1, z[(jj + 1) * zs], cur[(jj + 1) * SF_ENVS + lane]);
    }
    if (pf.nb & 1) t2_cmac_sub32(acc, z[(pf.nb - 1) * zs], cur[(pf.nb - 1) * SF_ENVS + lane]);
    return make_float2(acc.x + a1.x, acc.y + a1.y);
  };

  uint32_t act_phase = 0;
  for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int e_raw = P.e_lo + tile * SF_ENVS + lane;
    const bool valid = e_raw < P.e_hi;
    const int e = valid ? e_raw : P.e_hi - 1;

    // warm-start voltage of my branch and the episode returns: issued now, used after the components
    double2 up = make_double2((double)cst.x, (double)cst.y);
    if (pf.warm_start && b < pf.nb) up = pf.u_state[(size_t)b * E + e];
    double er0 = 0.0;
    if (w < pc.A) er0 = pf.ep_ret[(size_t)w * E + e];
    if (w < 3) sDmax[w * SF_ENVS + lane] = 0;

    if (first_tile) mbar_wait(&mbar_ev, 0);            // event row has landed
    if (tile_in_smem(tile)) {                          // CTA uniform
      mbar_wait(&mbar_act, act_phase);
      act_phase ^= 1u;
      io.actions = sAct; io.aE = SF_ENVS; io.ae0 = P.e_lo + tile * SF_ENVS;
    } else {
      io.actions = static_cast<const IoT*>(pc.actions); io.aE = E; io.ae0 = 0;
    }
    SF_STAMP(3);

    // ---- components: warp w steps components w, w + 16, ... of every env of the tile
    for (int ci = w; ci < P.C; ci += SF_WARPS) {
      const pgw_component c = comps[ci];
      double pw = 0.0, rw = 0.0;
      if (valid) {
        switch (c.type) {
          case PGW_STORAGE: storage_step(c, io, e, pw); break;
          case PGW_PV: pv_step(c, io, e, pw, rw); break;
          case PGW_EV: ev_step(c, io, e, pw, rw); break;
          case PGW_BUILDING: building_step_fast(c, io, e, pw, rw); break;
          default: break;
        }
      }
      sCp[ci * SF_ENVS + lane] = pw;
      sCr[ci * SF_ENVS + lane] = rw;
    }
    if (w == 0 && valid) pc.done[e] = drow[0] != 0.0 ? 1 : 0;
    SF_STAMP(4);
    __syncthreads();
    // Host-buffer steps run as a chain of env chunks (programmatic dependent launches): this CTA
    // has read the actions of its last tile, the next chunk may start reading its own while this
    // one's observations drain over the other direction of the link.
    if (P.pdl_trigger && tile + (int)gridDim.x >= tiles) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (w == 1) fetch_actions(tile + (int)gridDim.x);  // the staging area is free again
    SF_STAMP(5);

    // ---- agents: real power (base.py:51-55; summed in component order from 0.0 like the
    //      reference), kept for the power flow; the reward waits for the penalty
    double rew0 = 0.0;
    for (int a = w; a < pc.A; a += SF_WARPS) {
      const pgw_agent ag = agents[a];
      double pa = 0.0, ra = 0.0;
      for (int ci = ag.comp_begin; ci < ag.comp_end; ++ci) {
        pa += sCp[ci * SF_ENVS + lane];
        ra += sCr[ci * SF_ENVS + lane];
      }
      if (valid) pc.agent_p[(size_t)a * E + e] = pa;
      if (a == w) rew0 = ra;
    }

    // ---- nominal power of my branch: base load of the event + the agents on its load
    //      (multiagent_env.py:171-181: summed per load name in agent order; opendss.py:128)
    float sr = 0.f, si = 0.f;
    double2 s64 = make_double2(0.0, 0.0);
    float2 dprev = make_float2(0.f, 0.f), cur = make_float2(0.f, 0.f);
    if (b < pf.nb) {
      const int l = bload[b];
      double ctl = 0.0;
      for (int q = lptr[l]; q < lptr[l + 1]; ++q) {
        const pgw_agent ag = agents[lidx[q]];
        double pa = 0.0;
        for (int ci = ag.comp_begin; ci < ag.comp_end; ++ci) pa += sCp[ci * SF_ENVS + lane];
        ctl += pa;
      }
      const double kw = drow[2 + l] + ctl, kvar = drow[2 + pf.nl + l];
      const float sh = share[b] * xs;
      sr = (float)kw * sh;
      si = (float)kvar * sh;
      s64 = make_double2(kw * kp.share[b], kvar * kp.share[b]);
      dprev = make_float2(((float)up.x - cst.x) * (1.f / ds1), ((float)up.y - cst.y) * (1.f / ds1));
      t2_current<ANY_M5>(cst, gh, dprev.x, dprev.y, ds1, sr, si, cur.x, cur.y);
      sI32[b * SF_ENVS + lane] = cur;
    }
    __syncthreads();
    SF_STAMP(6);

    // ---- fixed point: iteration `it` reads the currents of parity (it - 1) & 1 and writes those
    //      of parity it & 1 (one barrier per iteration); the convergence maxima rotate over three
    //      slots, so that warp 0 can clear the next one before the barrier: every thread has read
    //      it (two iterations ago) before it arrived at the previous barrier
    int it = 0, my_it = 0;
    bool conv = !valid, conv_ok = true;
    while (true) {
      ++it;
      const int slot = it % 3;
      if (w == 0) sDmax[((it + 1) % 3) * SF_ENVS + lane] = 0;
      if (b < pf.nb) {
        const float2 d = zdot(make_float2(0.f, 0.f), z32 + b, 16, sI32 + ((it - 1) & 1) * 16 * SF_ENVS);
        const float2 dn = make_float2(d.x * rds1, d.y * rds1);
        const float dd = fmaxf(fabsf(dn.x - dprev.x), fabsf(dn.y - dprev.y));
        atomicMax(&sDmax[slot * SF_ENVS + lane], __float_as_int(dd));
        if (!conv) t2_current<ANY_M5>(cst, gh, dn.x, dn.y, ds1, sr, si, cur.x, cur.y);   // converged envs keep theirs
        sI32[((it & 1) * 16 + b) * SF_ENVS + lane] = cur;
        dprev = dn;
      }
      __syncthreads();
      if (!conv) {
        const float d = __int_as_float(sDmax[slot * SF_ENVS + lane]);
        conv_ok = d < tol_s;
        conv = conv_ok || it >= pf.max_iter;
        my_it = it;
      }
      if (__all_sync(0xffffffffu, conv ? 1 : 0) != 0) break;
    }

    SF_STAMP(7);
    [[maybe_unused]] const int it_stamp = it;
    const float2* i_fin = sI32 + (it & 1) * 16 * SF_ENVS;   // the fixed point's final currents
    // ---- float64 polish of my branch voltage
    const bool polish = t.polish > 0 && pf.reward_hook;
    double2 u64 = make_double2(kp.u0[b].x + (double)dprev.x * (double)ds1,
                               kp.u0[b].y + (double)dprev.y * (double)ds1);
    const bool my_row = ((kp.rows >> b) & 1u) != 0u;
    if (polish) {
      const int sweeps = t.polish + ((kp.rows != 0u || t.polish_row >= 0) ? 1 : 0);
      // Sweep 0 in float32: the fixed point's iteration once more, from its last drop, with
      // correctly rounded reciprocals in the currents, into the other parity's array (free again:
      // its last reader passed the loop's last barrier).  A full sweep only has to take every branch voltage from the fixed
      // point's ~1e-7 p.u. to ~1e-8: it feeds the currents of the next sweep, whose rows the rewards
      // read in float64, and a sweep contracts the error by more than 10x.  Float32 currents are
      // half the shared-memory traffic of the float64 sweep (every thread reads all currents of
      // its env: 14 warps x 14 x 512 B was the sweep's bound) and the FMAs run on the FP32 pipe.
      {
        float2* i_pre = sI32 + ((it + 1) & 1) * 16 * SF_ENVS;
        if (b < pf.nb) {
          float x, y;
          t2_current32<ANY_M5>(cst, gh, dprev.x, dprev.y, ds1, sr, si, x, y);
          i_pre[b * SF_ENVS + lane] = make_float2(x, y);
        }
        __syncthreads();
        if (b < pf.nb) {
          const float2 d = zdot(make_float2(0.f, 0.f), z32 + b, 16, i_pre);
          u64 = make_double2(kp.u0[b].x + (double)d.x, kp.u0[b].y + (double)d.y);
          if (t.polish == 1 && valid) pf.u_state[(size_t)b * E + e] = u64;
        }
      }
#pragma unroll 1
      for (int sweep = 1; sweep < sweeps; ++sweep) {
        __syncthreads();                               // everyone has read the previous currents
        if (b < pf.nb) sI64[b * SF_ENVS + lane] = t2_current64(kp.model[b], s64, u64, kp.vlo2[b], kp.vhi2[b]);
        __syncthreads();
        if (b < pf.nb && (sweep < t.polish || my_row)) {
          double2 a0 = kp.u0[b], a1 = make_double2(0.0, 0.0);
#pragma unroll 2
          for (int jj = 0; jj + 1 < pf.nb; jj += 2) {
            t2_cmac_sub64(a0, kp.zT[jj * 16 + b], sI64[jj * SF_ENVS + lane]);
            t2_cmac_sub64(a1, kp.zT[(jj + 1) * 16 + b], sI64[(jj + 1) * SF_ENVS + lane]);
          }
          if (pf.nb & 1) t2_cmac_sub64(a0, kp.zT[(pf.nb - 1) * 16 + b], sI64[(pf.nb - 1) * SF_ENVS + lane]);
          u64 = make_double2(a0.x + a1.x, a0.y + a1.y);
        }
        if (sweep + 1 == t.polish && valid && b < pf.nb) pf.u_state[(size_t)b * E + e] = u64;
      }
    } else if (valid && b < pf.nb) {
      pf.u_state[(size_t)b * E + e] = u64;
    }

    SF_STAMP(8);
    // ---- node magnitudes: my branch's wye-load node, then my slots of the expansion
    float vmn = 3.0e38f, vmx = -3.0e38f;
    if (b < pf.nb) {
      const int n = dnode[b];
      if (n >= 0) {
        const double m2 = u64.x * u64.x + u64.y * u64.y;
        double mag;
        if (polish) {
          mag = sqrt(m2) * kp.dscale[b];
        } else {
          const float m2f = (float)m2;
          mag = (double)(m2f * t2_rsqrt(fmaxf(m2f, 1e-30f)) * dscale[b]);
        }
        vmn = vmx = (float)mag;
        sVn[b * SF_ENVS + lane] = mag;
        if (valid) pf.vmag[(size_t)n * E + e] = mag;
      }
    }
    for (int cc = 0; cc < t.ncc; ++cc) {
      const int slot = 16 * cc + b;                    // warp uniform
      if (slot < t.nx) {
        const int n = xnode[slot];
        if (n >= 0) {
          // - Znb i summed from zero (terms of the size of a drop), then w added once
          const float2 dv = zdot(make_float2(0.f, 0.f), xz + slot, 16 * t.ncc, i_fin);
          const float2 wv = wx[slot];
          const float vr = wv.x + dv.x, vi = wv.y + dv.y;
          const float m2 = fmaf(vr, vr, vi * vi);
          const float mag = m2 * t2_rsqrt(fmaxf(m2, 1e-30f));
          vmn = fminf(vmn, mag);
          vmx = fmaxf(vmx, mag);
          if (valid) pf.vmag[(size_t)n * E + e] = (double)mag;
        }
      }
    }
    sVmn[w * SF_ENVS + lane] = vmn;
    sVmx[w * SF_ENVS + lane] = vmx;
    __syncthreads();                                   // magnitudes (global) and partials visible
    SF_STAMP(9);

    // Penalty node that is not a wye-load node: its row of the last sweep from the currents
    // still in shared memory.
    double v_row = 0.0;
    const bool have_row = polish && t.polish_row >= 0;
    if (have_row) {
      const double2* wv = reinterpret_cast<const double2*>(pf.blob + pf.off_w);
      const double2* zn = reinterpret_cast<const double2*>(pf.blob + pf.off_znbT);
      double2 v = wv[t.polish_row];
      for (int jj = 0; jj < pf.nb; ++jj)
        t2_cmac_sub64(v, zn[(size_t)jj * pf.nnp + t.polish_row], sI64[jj * SF_ENVS + lane]);
      v_row = sqrt(v.x * v.x + v.y * v.y);
      if (valid && w == 0) pf.vmag[(size_t)t.polish_row * E + e] = v_row;
    }
    if (valid) {
      double pen_share = 0.0, viol = 0.0;
      if (pf.punit != 0.0) {
        const double v = have_row ? v_row
                                  : (t.pen_slot >= 0 ? sVn[t.pen_slot * SF_ENVS + lane]
                                                     : pf.vmag[(size_t)pf.penalty_node * E + e]);
        viol = fmax(0.0, fmax(pf.pvlo - v, v - pf.pvhi));                 // train.py:71-88
        pen_share = (viol * pf.punit) / (double)pf.A;                     // train.py:56-61
      }
      if (w == 0) {
        float mn = sVmn[lane], mx = sVmx[lane];
#pragma unroll
        for (int q = 1; q < SF_WARPS; ++q) {
          mn = fminf(mn, sVmn[q * SF_ENVS + lane]);
          mx = fmaxf(mx, sVmx[q * SF_ENVS + lane]);
        }
        pf.vmin[e] = (double)mn;
        pf.vmax[e] = (double)mx;
        pf.iters[e] = conv_ok ? my_it : -my_it;
        pf.viol[e] = viol;
      }
      // every agent: bus voltage, reward (minus the shared penalty), episode return
      for (int a = w; a < pc.A; a += SF_WARPS) {
        const size_t ae = (size_t)a * E + e;
        double ra = rew0, er = er0;
        if (a != w) {
          const pgw_agent ag = agents[a];
          ra = 0.0;
          for (int ci = ag.comp_begin; ci < ag.comp_end; ++ci) ra += sCr[ci * SF_ENVS + lane];
          er = pf.ep_ret[ae];
        }
        const int node = anode[a];
        double vb = 1.0;
        if (node >= 0)
          vb = (have_row && node == t.polish_row) ? v_row
               : (aslot[a] >= 0 ? sVn[aslot[a] * SF_ENVS + lane] : pf.vmag[(size_t)node * E + e]);
        const double r = pf.reward_hook ? ra - pen_share : ra;
        pf.vbus[ae] = vb;
        pc.rew[ae] = r;
        pf.rew_copy[ae] = r;
        pf.ep_ret[ae] = er + r;
      }
    }
    __syncthreads();                                   // shared arrays are reused by the next tile
    SF_STAMP(10);
#ifdef PGW_PHASE_TIMERS
    if (pf.phase_clk != nullptr && threadIdx.x == 0 && SF_STAMP_TILE) pf.phase_clk[(size_t)(blockIdx.x + P.e_lo / SF_ENVS) * 16 + 11] = it_stamp;
#endif
    first_tile = false;
  }

  if (tid == 0) {
    if (!host_event) clock_advance_if_last(my_ticket, pc.ticket, pc.clock, clk, P.tickets);
    else if (blockIdx.x == 0) *pc.clock = event;       // nobody reads it in this mode: any CTA may publish
  }
#ifdef PGW_PHASE_TIMERS
  if (pf.phase_clk != nullptr && threadIdx.x == 0) {
    pf.phase_clk[(size_t)(blockIdx.x + P.e_lo / SF_ENVS) * 16 + 14] = clock64();
    pf.phase_clk[(size_t)(blockIdx.x + P.e_lo / SF_ENVS) * 16 + 13] = (long long)global_timer_ns();
  }
#endif
}

bool is_step_fused_kernel(const void* func) {
  return func == (const void*)step_fused_kernel<false, false> || func == (const void*)step_fused_kernel<true, false> ||
         func == (const void*)step_fused_kernel<false, true> || func == (const void*)step_fused_kernel<true, true>;
}

size_t step_fused_smem_bytes(const FusedParams& P) { return sf_layout(P).total; }

int step_fused_tiles(int envs) { return (envs + SF_ENVS - 1) / SF_ENVS; }

cudaError_t launch_step_fused(const FusedParams& P, int grid, cudaStream_t s, bool programmatic) {
  auto kern = P.c.io32 ? (P.f.tc2.any_m5 ? step_fused_kernel<true, true> : step_fused_kernel<false, true>)
                       : (P.f.tc2.any_m5 ? step_fused_kernel<true, false> : step_fused_kernel<false, false>);
  const size_t smem = step_fused_smem_bytes(P);
  cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(SF_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = programmatic ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, P);
}

}  // namespace pgw
