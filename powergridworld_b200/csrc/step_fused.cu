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
// * Power flow: the row products of u <- u0 - Zbb i(u) run on warp-level mma.sync.m16n8k16 with
//   the split-FP16 operands of powerflow_tc2.cu (currents x xscale and Zbb x sb1 as FP16 hi + lo,
//   hi.hi + hi.lo + lo.hi accumulated in FP32): the tile is two m-tiles of 16 envs, the realified
//   Zbb four n-tiles of 4 branches with (Re, Im) interleaved, so warp 4m + j's D fragment holds
//   the complex drop of branch 4j + lane % 4 for two envs -- the input of the load model, in
//   registers.  The currents go back as FP16 hi / lo A operands (double-buffered by iteration
//   parity, read by ldmatrix), the warps of an m-tile meet at a named barrier of their own, and
//   each m-tile leaves the loop when its 16 envs have converged (max |d drop| per env through a
//   shared-memory atomicMax; converged envs freeze their currents).  No tcgen05: at 32 envs a
//   tile, its commit / mbarrier / TMEM hand-offs were the latency (DESIGN.md section 4.3d).
// * Polish: the fixed point's iteration once more with correctly rounded currents (one more MMA
//   product), then float64 sweeps u <- u0 - Zbb i(u) on the SIMT pipe, one branch per thread
//   (the env's currents through shared memory), spread over 16 warps and -- with 32-env tiles --
//   over every SM of the GPU: ~0.4 us per sweep at 4096 envs instead of ~3 us in the 128-env
//   tiles of powerflow_tc2.cu.
// * Expansion v = w - Znb i for the nodes that are not a wye-load node: the same MMA product
//   against Znb x sb2 from the fixed point's final currents, n-tiles of 4 node slots.
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

// The fixed point's A operands: per iteration parity and m-tile (16 envs), 16 env rows of
// [hi: 16 branches x (Re, Im) FP16 | lo: the same | 16 bytes of padding].  The 144-byte row
// stride puts the 8 rows of every ldmatrix phase, and the 8 env groups of every current store,
// on distinct banks.
constexpr int SF_AROW = 144;
constexpr int SF_ATILE = 16 * SF_AROW;

struct SfLayout {                                      // byte offsets into dynamic shared memory
  uint32_t tab, ftab, blob, drow, irow, ia, ld, i64, dmax, part, vn, cp, cr, act, total;
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
  L.ia = take(2u * 2u * SF_ATILE);                     // fixed-point A operands, [parity][m-tile]
  L.ld = take(16u * SF_ENVS * 16u);                    // {sr, si, drop} of each branch, [k][env] float4
  L.i64 = take(16u * SF_ENVS * 16u);                   // currents of a polish sweep
  L.dmax = take(9u * SF_ENVS * 4u);                    // convergence maxima [2][env][4] + the iterations
  L.part = take(2u * 24u * SF_ENVS * 4u);              // min / max |v| partials: 16 warps, 8 n-tiles
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

__device__ __forceinline__ void sf_ldsm_x4(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(saddr)
               : "memory");
}

// d += a b: m16n8k16, FP16 operands, FP32 accumulators
__device__ __forceinline__ void sf_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// The A fragments of one m-tile: 16 envs x 16 branch currents (Re, Im), hi and lo, both k-steps
struct SfA {
  uint32_t h0[4], l0[4], h1[4], l1[4];
};

// The shared-memory address lane `lane` hands to ldmatrix.x4 for parity 0 of m-tile m: row
// (lane & 7) + 8 ((lane >> 3) & 1) of the 16 x 16 block, 16-byte column half lane >> 4
__device__ __forceinline__ uint32_t sf_a_lane(const uint32_t* sIA, int m, int lane) {
  return smem_u32(sIA) + (uint32_t)m * SF_ATILE +
         (uint32_t)((((lane >> 3) & 1) * 8 + (lane & 7)) * SF_AROW + (lane >> 4) * 16);
}

__device__ __forceinline__ void sf_load_a(SfA& A, uint32_t a) {
  sf_ldsm_x4(A.h0, a);
  sf_ldsm_x4(A.l0, a + 64);
  sf_ldsm_x4(A.h1, a + 32);
  sf_ldsm_x4(A.l1, a + 96);
}

// The product of an m-tile's currents with n-tile (bk0, bk1) of a B image ({hi b0, hi b1, lo b0,
// lo b1} of k-steps 0 / 1): hi.hi + hi.lo + lo.hi, the small terms first, one accumulator chain per
// k-step.  d = {Re, Im} of output 4j + tq for env row g, then for env row g + 8.
__device__ __forceinline__ void sf_product(float (&d)[4], const SfA& A, uint4 bk0, uint4 bk1) {
  float d0[4] = {0.f, 0.f, 0.f, 0.f}, d1[4] = {0.f, 0.f, 0.f, 0.f};
  sf_mma(d0, A.l0, bk0.x, bk0.y);
  sf_mma(d1, A.l1, bk1.x, bk1.y);
  sf_mma(d0, A.h0, bk0.z, bk0.w);
  sf_mma(d1, A.h1, bk1.z, bk1.w);
  sf_mma(d0, A.h0, bk0.x, bk0.y);
  sf_mma(d1, A.h1, bk1.x, bk1.y);
#pragma unroll
  for (int q = 0; q < 4; ++q) d[q] = d0[q] + d1[q];
}

// A current (scaled by xscale) as its FP16 hi / lo (Re, Im) pairs into an A row, at word q of each half
__device__ __forceinline__ void sf_put_current(uint32_t* row, int q, float2 c) {
  const uint32_t h = t2_pack(c.x, c.y);
  const float2 back = __half22float2(*reinterpret_cast<const __half2*>(&h));
  row[q] = h;
  row[16 + q] = t2_pack(c.x - back.x, c.y - back.y);
}

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
  unsigned char* sBlob = sf_smem + L.blob;
  double* drow = reinterpret_cast<double*>(sf_smem + L.drow);
  int32_t* irow = reinterpret_cast<int32_t*>(sf_smem + L.irow);
  uint32_t* sIA = reinterpret_cast<uint32_t*>(sf_smem + L.ia);     // [parity][m-tile][16 rows][36 words]
  float4* sLd = reinterpret_cast<float4*>(sf_smem + L.ld);         // [16][env]
  double2* sI64 = reinterpret_cast<double2*>(sf_smem + L.i64);
  int* sDmax = reinterpret_cast<int*>(sf_smem + L.dmax);           // [parity][env][n-tile] float bits
  int* sIters = sDmax + 2 * SF_ENVS * 4;                           // [env]: iterations, < 0 not converged
  float* sVmn = reinterpret_cast<float*>(sf_smem + L.part);        // [16][env]
  float* sVmx = sVmn + 16 * SF_ENVS;
  float* sXmn = sVmx + 16 * SF_ENVS;                               // [8][env]: the expansion's n-tile columns
  float* sXmx = sXmn + 8 * SF_ENVS;
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
  const float tol_s = t.tol / ds1;
  const float4 cst = t2_cst(kc, b);
  const float2 gh = ANY_M5 ? t2_gh(kc, b) : make_float2(1.f, 0.f);

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
    // (the padded branches b >= nb: zero power, zero current, zero drop)
    double2 s64 = make_double2(0.0, 0.0);
    {
      float sr = 0.f, si = 0.f;
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
      }
      sLd[b * SF_ENVS + lane] = make_float4(sr, si, dprev.x, dprev.y);
      sf_put_current(sIA + (lane >> 4) * (SF_ATILE / 4) + (lane & 15) * (SF_AROW / 4), b, cur);
    }
    __syncthreads();
    SF_STAMP(6);

    // ---- fixed point on the tensor cores (mma.sync): warp 4m + j, m < 2, j < 4, computes the drops
    //      of m-tile m (envs 16m .. 16m + 15) and n-tile j (branches 4j .. 4j + 3); thread (g, tq) =
    //      (lane / 4, lane % 4) holds branch 4j + tq of envs 16m + g and 16m + g + 8 in its D
    //      fragment, and runs the load model of both.  Iteration `it` reads the A operands of parity
    //      (it - 1) & 1 and writes those of parity it & 1; the m-tile's four warps meet at a named
    //      barrier of their own, and each m-tile leaves the loop when its 16 envs have converged.
    //      The convergence maxima are double-buffered by parity too: a slot is written again two
    //      iterations later, after every thread of the m-tile has read it and arrived at the barrier
    //      in between.  Warps 8 .. 15 wait at the barrier after the loop.
    const bool polish = t.polish > 0 && pf.reward_hook;
    if (w < 8) {
      const int m = w >> 2, j = w & 3, g = lane >> 2, tq = lane & 3;
      const int kb = 4 * j + tq;                       // my branch
      const bool active = kb < pf.nb;
      const int r0 = 16 * m + g, r1 = r0 + 8;          // my env rows of the tile
      const float4 c4 = t2_cst(kc, kb);
      const float2 g2 = ANY_M5 ? t2_gh(kc, kb) : make_float2(1.f, 0.f);
      const uint4* bz = reinterpret_cast<const uint4*>(sf_smem + L.ftab + t.f_xz) + (j * 32 + lane) * 2;
      const uint4 bk0 = bz[0], bk1 = bz[1];            // k-steps 0 / 1: {hi b0, hi b1, lo b0, lo b1}
      const float4 l0 = sLd[kb * SF_ENVS + r0], l1 = sLd[kb * SF_ENVS + r1];
      float2 dp0 = make_float2(l0.z, l0.w), dp1 = make_float2(l1.z, l1.w);
      float2 cu0 = make_float2(0.f, 0.f), cu1 = make_float2(0.f, 0.f);
      if (active) {                                    // the currents of parity 0, as the writer computed them
        t2_current<ANY_M5>(c4, g2, dp0.x, dp0.y, ds1, l0.x, l0.y, cu0.x, cu0.y);
        t2_current<ANY_M5>(c4, g2, dp1.x, dp1.y, ds1, l1.x, l1.y, cu1.x, cu1.y);
      }
      bool cv0 = e_raw - lane + r0 >= P.e_hi, cv1 = e_raw - lane + r1 >= P.e_hi;   // rows past the batch
      bool ok0 = true, ok1 = true;
      int it0 = 0, it1 = 0;
      const uint32_t a_lane = sf_a_lane(sIA, m, lane);
      uint32_t* my_row0 = sIA + m * (SF_ATILE / 4) + g * (SF_AROW / 4);
      int it = 0;
      while (true) {
        ++it;
        int* dmax = sDmax + (it & 1) * SF_ENVS * 4;
        SfA A;
        sf_load_a(A, a_lane + (uint32_t)((it - 1) & 1) * (2 * SF_ATILE));
        // the scaled drop: (x xscale) (Zbb x sb1) = drop / descale1
        float d[4];
        sf_product(d, A, bk0, bk1);
        const float2 dn0 = make_float2(d[0], d[1]), dn1 = make_float2(d[2], d[3]);
        // max |d drop| (float bits: non-negative floats order as ints) over the quad's 4 branches,
        // then over the m-tile's 4 warps from [env][n-tile] after the barrier
        int dd0 = __float_as_int(fmaxf(fabsf(dn0.x - dp0.x), fabsf(dn0.y - dp0.y)));
        int dd1 = __float_as_int(fmaxf(fabsf(dn1.x - dp1.x), fabsf(dn1.y - dp1.y)));
        dd0 = max(dd0, __shfl_xor_sync(0xffffffffu, dd0, 1));
        dd1 = max(dd1, __shfl_xor_sync(0xffffffffu, dd1, 1));
        dd0 = max(dd0, __shfl_xor_sync(0xffffffffu, dd0, 2));
        dd1 = max(dd1, __shfl_xor_sync(0xffffffffu, dd1, 2));
        if (tq < 2) dmax[(tq == 0 ? r0 : r1) * 4 + j] = tq == 0 ? dd0 : dd1;
        if (active) {                                  // converged envs keep their currents
          if (!cv0) t2_current<ANY_M5>(c4, g2, dn0.x, dn0.y, ds1, l0.x, l0.y, cu0.x, cu0.y);
          if (!cv1) t2_current<ANY_M5>(c4, g2, dn1.x, dn1.y, ds1, l1.x, l1.y, cu1.x, cu1.y);
        }
        uint32_t* row = my_row0 + (it & 1) * (SF_ATILE / 2);
        sf_put_current(row, kb, cu0);
        sf_put_current(row + 8 * (SF_AROW / 4), kb, cu1);
        dp0 = dn0;
        dp1 = dn1;
        asm volatile("bar.sync %0, 128;" ::"r"(1 + m) : "memory");
        if (!cv0) {
          const int4 q = reinterpret_cast<const int4*>(dmax)[r0];
          ok0 = __int_as_float(max(max(q.x, q.y), max(q.z, q.w))) < tol_s;
          cv0 = ok0 || it >= pf.max_iter;
          it0 = it;
        }
        if (!cv1) {
          const int4 q = reinterpret_cast<const int4*>(dmax)[r1];
          ok1 = __int_as_float(max(max(q.x, q.y), max(q.z, q.w))) < tol_s;
          cv1 = ok1 || it >= pf.max_iter;
          it1 = it;
        }
        if (__all_sync(0xffffffffu, (cv0 && cv1) ? 1 : 0) != 0) break;
      }
      if (polish) {
        // Sweep 0 of the polish, float32: the fixed point's iteration once more, from its last drop,
        // with correctly rounded reciprocals in the currents (A operands of parity 1, free: the
        // m-tile's last reads of it were before the loop's last barrier).  A full sweep only has
        // to take every branch voltage from the fixed point's ~1e-7 p.u. to ~1e-8: it feeds the
        // currents of the next sweep, whose rows the rewards read in float64, and a sweep
        // contracts the error by more than 10x.  Its drops (p.u.) go to the hand-over below.
        float2 c0 = make_float2(0.f, 0.f), c1 = make_float2(0.f, 0.f);
        if (active) {
          t2_current32<ANY_M5>(c4, g2, dp0.x, dp0.y, ds1, l0.x, l0.y, c0.x, c0.y);
          t2_current32<ANY_M5>(c4, g2, dp1.x, dp1.y, ds1, l1.x, l1.y, c1.x, c1.y);
        }
        uint32_t* row = my_row0 + SF_ATILE / 2;
        sf_put_current(row, kb, c0);
        sf_put_current(row + 8 * (SF_AROW / 4), kb, c1);
        asm volatile("bar.sync %0, 128;" ::"r"(1 + m) : "memory");
        SfA A;
        sf_load_a(A, a_lane + 2 * SF_ATILE);
        float d[4];
        sf_product(d, A, bk0, bk1);
        dp0 = make_float2(d[0] * ds1, d[1] * ds1);
        dp1 = make_float2(d[2] * ds1, d[3] * ds1);
      }
      // hand-over to the one-branch-per-thread phases: the last drops (scaled; p.u. after the
      // pre-sweep), the final currents, the iterations
      if (active) {
        reinterpret_cast<float2*>(&sLd[kb * SF_ENVS + r0])[1] = dp0;
        reinterpret_cast<float2*>(&sLd[kb * SF_ENVS + r1])[1] = dp1;
      }
      sf_put_current(my_row0, kb, cu0);                // parity 0: the expansion's A operands
      sf_put_current(my_row0 + 8 * (SF_AROW / 4), kb, cu1);
      if (j == 0 && tq == 0) sIters[r0] = ok0 ? it0 : -it0;
      if (j == 0 && tq == 1) sIters[r1] = ok1 ? it1 : -it1;
    }
    __syncthreads();
    SF_STAMP(7);
#ifdef PGW_PHASE_TIMERS
    int it_stamp = 0;                                  // the CTA's loop count: its slowest env
    if (tid == 0)
      for (int r = 0; r < SF_ENVS; ++r) it_stamp = max(it_stamp, abs(sIters[r]));
#endif
    // ---- float64 polish of my branch voltage, from the pre-sweep's drop (or the fixed point's)
    const float4 ld = sLd[b * SF_ENVS + lane];
    double2 u64 = polish ? make_double2(kp.u0[b].x + (double)ld.z, kp.u0[b].y + (double)ld.w)
                         : make_double2(kp.u0[b].x + (double)ld.z * (double)ds1,
                                        kp.u0[b].y + (double)ld.w * (double)ds1);
    const bool my_row = ((kp.rows >> b) & 1u) != 0u;
    if (polish) {
      const int sweeps = t.polish + ((kp.rows != 0u || t.polish_row >= 0) ? 1 : 0);
      if (t.polish == 1 && valid && b < pf.nb) pf.u_state[(size_t)b * E + e] = u64;
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
    sVmn[w * SF_ENVS + lane] = vmn;
    sVmx[w * SF_ENVS + lane] = vmx;
    // Expansion v = w - Znb i on mma.sync from the fixed point's final currents (the A operands of
    // parity 0): warp w takes m-tile w / 8 and the n-tiles (4 slots each) w % 8, w % 8 + 8, ...;
    // thread (g, tq) gets slot 4 nt + tq of envs 16m + g and 16m + g + 8.  - Znb i is summed from
    // zero (terms of the size of a drop), then w is added once.
    {
      const int m = w >> 3, g = lane >> 2, tq = lane & 3;
      const int r0 = 16 * m + g, r1 = r0 + 8;
      const int e0 = e_raw - lane + r0, e1 = e0 + 8;
      SfA A;
      sf_load_a(A, sf_a_lane(sIA, m, lane));
      float mn0 = 3.0e38f, mx0 = -3.0e38f, mn1 = 3.0e38f, mx1 = -3.0e38f;
      for (int nt = w & 7; nt < 4 * t.ncc; nt += 8) {
        const uint4* bx = reinterpret_cast<const uint4*>(sf_smem + L.ftab + t.f_xz) + ((4 + nt) * 32 + lane) * 2;
        float d[4];                                    // - Znb i x xscale x sb2
        sf_product(d, A, bx[0], bx[1]);
        const int slot = 4 * nt + tq;
        const int n = slot < t.nx ? xnode[slot] : -1;
        if (n >= 0) {
          const float2 wv = wx[slot];
          const float ds2 = t.descale2;               // a power of two: exact
          const float vr0 = wv.x + d[0] * ds2, vi0 = wv.y + d[1] * ds2;
          const float vr1 = wv.x + d[2] * ds2, vi1 = wv.y + d[3] * ds2;
          const float m20 = fmaf(vr0, vr0, vi0 * vi0), m21 = fmaf(vr1, vr1, vi1 * vi1);
          const float mag0 = m20 * t2_rsqrt(fmaxf(m20, 1e-30f)), mag1 = m21 * t2_rsqrt(fmaxf(m21, 1e-30f));
          mn0 = fminf(mn0, mag0);
          mx0 = fmaxf(mx0, mag0);
          mn1 = fminf(mn1, mag1);
          mx1 = fmaxf(mx1, mag1);
          if (e0 < P.e_hi) pf.vmag[(size_t)n * E + e0] = (double)mag0;
          if (e1 < P.e_hi) pf.vmag[(size_t)n * E + e1] = (double)mag1;
        }
      }
#pragma unroll
      for (int s = 1; s <= 2; s <<= 1) {
        mn0 = fminf(mn0, __shfl_xor_sync(0xffffffffu, mn0, s));
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, s));
        mn1 = fminf(mn1, __shfl_xor_sync(0xffffffffu, mn1, s));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, s));
      }
      if (tq == 0) { sXmn[(w & 7) * SF_ENVS + r0] = mn0; sXmx[(w & 7) * SF_ENVS + r0] = mx0; }
      if (tq == 1) { sXmn[(w & 7) * SF_ENVS + r1] = mn1; sXmx[(w & 7) * SF_ENVS + r1] = mx1; }
    }
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
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          mn = fminf(mn, sXmn[q * SF_ENVS + lane]);
          mx = fmaxf(mx, sXmx[q * SF_ENVS + lane]);
        }
        pf.vmin[e] = (double)mn;
        pf.vmax[e] = (double)mx;
        pf.iters[e] = sIters[lane];
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
