// Per-(env, agent) arithmetic of the component models, shared by the step and reset
// kernels of components.cu.  Everything here is float64 and is compiled with
// -fmad=false so that each operation rounds exactly like the NumPy/Python scalar
// arithmetic of the reference (the storage clamp, for instance, is discontinuous:
// a fused multiply-add could flip a branch the reference does not take).
//
// Reference semantics restated (paths relative to the reference root):
//   gridworld/utils.py:9-43                                  to_scaled / to_raw
//   gridworld/agents/energy_storage/energy_storage_env.py:100-157
//   gridworld/agents/pv/pv_profile_env.py:102-148
//   gridworld/agents/vehicles/ev_charging_env.py:135-264
//   gridworld/agents/buildings/five_zone_rom_env.py:147-335
//   gridworld/agents/buildings/five_zone_rom_dynamics.py:12-114
//   gridworld/base.py:114-156                                composite agent
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/pgw.h"

#if defined(__CUDACC__)
#define PGW_HD __host__ __device__ __forceinline__
#else
#define PGW_HD inline
#endif
#define PGW_RESTRICT __restrict__
#if defined(__CUDA_ARCH__)
#define PGW_POPC(x) __popc(x)
#define PGW_CTZ(x) (__ffs((int)(x)) - 1)
#else
#define PGW_POPC(x) __builtin_popcount(x)
#define PGW_CTZ(x) __builtin_ctz(x)
#endif
#if defined(__CUDACC__)
#define PGW_NO_UNROLL _Pragma("unroll 1")
#else
#define PGW_NO_UNROLL
#endif

namespace pgw {

// Per-thread scratch array: element i lives at p[i * stride].
struct Scratch {
  double* p;
  int stride;
  PGW_HD double& operator[](int i) const { return p[(size_t)i * stride]; }
};
constexpr int kScratchDoubles = 35;

// Everything one (env, agent) worker needs; all per-env arrays are rows x E.  ActT / ObsT: element
// types of the caller's action and observation arrays (double, or float for float32 I/O).  The
// arithmetic is float64 either way: actions are widened exactly where they are read (act_in),
// observations rounded to nearest where they are stored (obs_val).
template <class ActT, class ObsT>
struct AgentIOT {
  Scratch scr;
  int E;
  // The arrays never alias each other; telling the compiler lets it overlap the many
  // independent load -> divide -> store chains of one agent (the kernel is latency bound).
  const ActT* PGW_RESTRICT actions;     // [act_dim][aE], env e at column e - ae0 (unused at reset): the
  int aE, ae0;                          // caller's [act_dim][E] array (aE = E, ae0 = 0) or a tile of it
                                        // staged in shared memory (step_fused.cu)
  ObsT* PGW_RESTRICT obs;               // [obs_dim][E]
  double* PGW_RESTRICT sd;              // [sd_rows][E]
  uint32_t* PGW_RESTRICT si;            // [si_rows][E]
  const double* PGW_RESTRICT init_soc;  // [num_storage][E] or nullptr (reset only)
  int clip_init_soc;                    // 1: an explicit init_storage, clipped to the storage range
                                        // (energy_storage_env.py:88-89); 0: the values are the
                                        // reference's own draw, which it does not clip (:82-84)
  const double* PGW_RESTRICT vmin;      // [E]    lagged grid variables (previous solve) or nullptr
  const double* PGW_RESTRICT vmax;      // [E]
  const double* PGW_RESTRICT vbus;      // [A][E]
  const double* PGW_RESTRICT dpar;
  const int32_t* PGW_RESTRICT ipar;
  const double* PGW_RESTRICT drow;      // event row (doubles)
  const int32_t* PGW_RESTRICT irow;     // event row (int32)
};
using AgentIO = AgentIOT<double, double>;

PGW_HD double clip(double x, double lo, double hi) { return fmin(fmax(x, lo), hi); }

// action row `row` of env e, widened to double (exact for a float)
template <class IO>
PGW_HD double act_in(const IO& io, int row, int e) {
  return (double)io.actions[(size_t)row * io.aE + (e - io.ae0)];
}

// an observation value in the caller's element type: as computed, or rounded to the nearest float
PGW_HD double io_round(double v, const double*) { return v; }
PGW_HD float io_round(double v, const float*) {
#if defined(__CUDA_ARCH__)
  return __double2float_rn(v);
#else
  return static_cast<float>(v);
#endif
}
template <class IO>
PGW_HD auto obs_val(const IO& io, double v) { return io_round(v, io.obs); }

// x / d when r = RN(1/d) was computed on the host: one multiply plus one FMA-based
// correction (Markstein) returns the correctly rounded IEEE quotient, i.e. the same bits
// as the reference's division, at a third of the dependent latency of a full FP64
// divide.  fma() is explicit here; everything else in this file is compiled -fmad=false.
PGW_HD double div_by(double x, double d, double r) {
  const double q = x * r;
  const double rem = fma(-q, d, x);
  return fma(rem, r, q);
}

// utils.py:27-43
PGW_HD double to_raw(double y, double lo, double hi) {
  y = clip(y, -1.0, 1.0);
  return (y * (hi - lo) + (hi + lo)) / 2.0;
}
// utils.py:9-24; inv = RN(1 / (hi - lo))
PGW_HD double to_scaled(double x, double lo, double hi, double inv) {
  x = clip(x, lo, hi);
  return div_by(2.0 * x - (lo + hi), hi - lo, inv);
}

// ------------------------------------------------------------------ storage
PGW_HD double storage_obs(const pgw_component& c, const double* dp, double soc) {
  return (c.flags & PGW_F_RESCALE) ? to_scaled(soc, dp[0], dp[1], dp[7]) : soc;
}

template <class IO>
PGW_HD void storage_reset(const pgw_component& c, const IO& io, int e) {
  const double* dp = io.dpar + c.dpar_off;
  double* soc = io.sd + (size_t)c.sd_off * io.E + e;
  const int ord = io.ipar[c.ipar_off];
  const double init = io.init_soc != nullptr ? io.init_soc[(size_t)ord * io.E + e] : dp[6];
  *soc = (io.init_soc != nullptr && !io.clip_init_soc) ? init : clip(init, dp[0], dp[1]);   // :82-89
  io.obs[(size_t)c.obs_off * io.E + e] = obs_val(io, storage_obs(c, dp, *soc));
}

template <class IO>
PGW_HD void storage_step(const pgw_component& c, const IO& io, int e, double& p_out) {
  const double* dp = io.dpar + c.dpar_off;
  const double lo = dp[0], hi = dp[1], eta_c = dp[2], eta_d = dp[3], pmax = dp[4], dt = dp[5];
  const double inv_eta_d = dp[8], inv_dt = dp[9];
  double a = act_in(io, c.act_off, e);
  if (c.flags & PGW_F_RESCALE) a = to_raw(a, -1.0, 1.0);
  double* soc_p = io.sd + (size_t)c.sd_off * io.E + e;
  double soc = *soc_p;
  double p = a * pmax;
  // validate_power :100-128 (the clamps omit the efficiencies, as in the reference)
  if (p > 0.0) {
    if (soc - div_by(p * dt, eta_d, inv_eta_d) < lo) p = div_by(fmax(soc - lo, 0.0), dt, inv_dt);
  } else if (p < 0.0) {
    if (soc - eta_c * p * dt > hi) p = div_by(-fmax(hi - soc, 0.0), dt, inv_dt);
  }
  if (p < 0.0) {
    soc -= eta_c * p * dt;
    soc = fmin(soc, hi);
  } else if (p > 0.0) {
    soc -= div_by(p * dt, eta_d, inv_eta_d);
    soc = fmax(soc, lo);
  }
  *soc_p = soc;
  io.obs[(size_t)c.obs_off * io.E + e] = obs_val(io, storage_obs(c, dp, soc));
  p_out = -p;
}

// ------------------------------------------------------------------ PV
template <class IO>
PGW_HD void pv_obs(const pgw_component& c, const IO& io, int e, double raw_power) {
  const double* dp = io.dpar + c.dpar_off;
  const bool rs = (c.flags & PGW_F_RESCALE) != 0;
  io.obs[(size_t)c.obs_off * io.E + e] =
      obs_val(io, rs ? to_scaled(raw_power, dp[0], dp[1], dp[4]) : raw_power);
  if (c.flags & PGW_F_GRID_AWARE) {
    const double v = io.vmin[e];
    io.obs[(size_t)(c.obs_off + 1) * io.E + e] = obs_val(io, rs ? to_scaled(v, dp[2], dp[3], dp[5]) : v);
  }
}

template <class IO>
PGW_HD void pv_step(const pgw_component& c, const IO& io, int e, double& p_out,
                    double& rew) {
  double a = act_in(io, c.act_off, e);
  if (c.flags & PGW_F_RESCALE) a = to_raw(a, 0.0, 1.0);
  const double raw_power = -io.drow[c.dtab_off];      // obs of the PRE-increment row (:143)
  pv_obs(c, io, e, raw_power);
  p_out = a * raw_power;
  rew = 0.0;
  if (c.flags & PGW_F_PV_VOLT_REWARD) {               // heterogeneous.py:46-52 (lagged vmin)
    const double v = io.vmin[e];
    const double viol = fmin(0.0, v - 0.95) + fmin(0.0, 1.05 - v);
    const double s = 1000.0 * viol;
    rew = -(s * s);
  }
}

// ------------------------------------------------------------------ EV station
// One pass over the vehicles parked at the event's time (the roster is shared by
// all envs, so the window is a per-event list; only the "energy > 0" part of the
// reference's charging set is per-env).  kwh = energy one vehicle may take now.
constexpr int kEvBatch = 8;   // vehicles whose energies are in flight together

struct EvTotals {
  double consumed, demand, deficit_sum, unserved;
  int active, n_deficit;
};

// The charging pass shared by the stock station and the Home-Steward charger: window of the
// event's evaluation time t_now, per-vehicle energy update, charging-set mask, unserved energy
// of the vehicles that left the window.
template <class IO>
PGW_HD EvTotals ev_charge_pass(const pgw_component& c, const IO& io, int e, double kwh) {
  const double* dp = io.dpar + c.dpar_off;
  const int32_t* ip = io.ipar + c.ipar_off;
  const int words = ip[1], cap = ip[2];
  const double rate = dp[0];
  const double* lh = io.drow + c.dtab_off + 2;         // [cap] hours left, by window slot
  const double* ilh = lh + cap;                        // [cap] 1 / hours left
  const int32_t* ir = io.irow + c.itab_off;
  const int n_win = ir[0], n_left = ir[1];
  const int32_t* win = ir + 2;
  const int32_t* left = ir + 2 + cap;
  double* energy = io.sd + (size_t)c.sd_off * io.E + e;
  uint32_t* mask = io.si + (size_t)c.si_off * io.E + e;

  EvTotals t;
  t.consumed = 0.0; t.demand = 0.0; t.deficit_sum = 0.0; t.unserved = 0.0;
  t.active = 0; t.n_deficit = 0;
  uint32_t word = 0;
  int cur_word = 0;
  for (int w = 0; w < words; ++w) mask[(size_t)w * io.E] = 0u;
  // Ascending vehicle index, kEvBatch vehicles per trip: their energies are loaded up front so
  // that as many independent HBM/L2 requests are in flight per thread (a vehicle's store can
  // never alias another vehicle's load, which the compiler cannot know).
  for (int k0 = 0; k0 < n_win; k0 += kEvBatch) {
    int idx[kEvBatch];
    double need4[kEvBatch];
#pragma unroll
    for (int j = 0; j < kEvBatch; ++j) {
      idx[j] = k0 + j < n_win ? win[k0 + j] : -1;
      need4[j] = idx[j] >= 0 ? energy[(size_t)idx[j] * io.E] : 0.0;
    }
#pragma unroll
    for (int j = 0; j < kEvBatch; ++j) {
      const int i = idx[j];
      const double need = need4[j];
      if (i < 0 || !(need > 0.0)) continue;             // :191
      if ((i >> 5) != cur_word) {
        if (word) mask[(size_t)cur_word * io.E] = word;
        cur_word = i >> 5;
        word = 0;
      }
      word |= 1u << (i & 31);
      ++t.active;
      t.demand += need;                                 // :210
      // hours left until the vehicle departs and the correctly rounded reciprocal, both compiled
      // per window slot into the event row: need / left_h becomes a multiply + FMA correction
      const double left_h = lh[k0 + j];
      if (left_h <= 0.0) continue;                      // :218-220
      t.deficit_sum += fmax(0.0, rate - div_by(need, left_h, ilh[k0 + j]));   // :221-223
      ++t.n_deficit;
      const double delta = fmin(kwh, need);             // :226-228
      energy[(size_t)i * io.E] = need - delta;
      t.consumed += delta;
    }
  }
  if (word) mask[(size_t)cur_word * io.E] = word;
  // :240-243 over window(k-1) \ window(k)
  for (int k = 0; k < n_left; ++k) t.unserved += energy[(size_t)left[k] * io.E];
  return t;
}

// The same pass for a station whose roster is PER ENV (PGW_F_EV_PER_ENV: every env instance of a
// randomised station samples its own vehicles, ev_charging_env.py:154-157): slot i of env e parks
// from floor(start) to floor(end) minutes, packed into the env's window word i; "parked at t" is
// evaluated per env (:186-190), the departed vehicles are old charging set \ new one (:194).
template <class IO>
PGW_HD EvTotals ev_charge_pass_env(const pgw_component& c, const IO& io, int e, double kwh) {
  const double* dp = io.dpar + c.dpar_off;
  const int32_t* ip = io.ipar + c.ipar_off;
  const int n = ip[0], words = ip[1];
  const double rate = dp[0], inv60 = dp[20];
  const double t_now = io.drow[c.dtab_off];
  double* energy = io.sd + (size_t)c.sd_off * io.E + e;
  uint32_t* mask = io.si + (size_t)c.si_off * io.E + e;
  const uint32_t* win = mask + (size_t)words * io.E;

  EvTotals t;
  t.consumed = 0.0; t.demand = 0.0; t.deficit_sum = 0.0; t.unserved = 0.0;
  t.active = 0; t.n_deficit = 0;
  uint32_t old_w[8], new_w[8];
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    old_w[w] = w < words ? mask[(size_t)w * io.E] : 0u;
    new_w[w] = 0u;
  }
  for (int i0 = 0; i0 < n; i0 += kEvBatch) {           // ascending slot index, loads batched
    uint32_t ww[kEvBatch];
    double need8[kEvBatch];
#pragma unroll
    for (int j = 0; j < kEvBatch; ++j) ww[j] = i0 + j < n ? win[(size_t)(i0 + j) * io.E] : 0xFFFF0000u;
#pragma unroll
    for (int j = 0; j < kEvBatch; ++j) {
      const bool parked = t_now >= (double)(ww[j] >> 16) && t_now <= (double)(ww[j] & 0xFFFFu);
      need8[j] = parked ? energy[(size_t)(i0 + j) * io.E] : 0.0;
    }
#pragma unroll
    for (int j = 0; j < kEvBatch; ++j) {
      const int i = i0 + j;
      const double need = need8[j];
      if (!(need > 0.0)) continue;                      // not parked, or :191
#pragma unroll
      for (int w = 0; w < 8; ++w)                       // (static indices: the words stay in registers)
        if (w == (i >> 5)) new_w[w] |= 1u << (i & 31);
      ++t.active;
      t.demand += need;                                 // :210
      const double left_h = div_by((double)(ww[j] & 0xFFFFu) - t_now, 60.0, inv60);   // :216
      if (left_h <= 0.0) continue;                      // :218-220
      t.deficit_sum += fmax(0.0, rate - need / left_h); // :221-223
      ++t.n_deficit;
      const double delta = fmin(kwh, need);             // :226-228
      energy[(size_t)i * io.E] = need - delta;
      t.consumed += delta;
    }
  }
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    if (w < words) {
      mask[(size_t)w * io.E] = new_w[w];
      uint32_t gone = old_w[w] & ~new_w[w];             // :240-243, ascending index
      while (gone) {
        const int bit = PGW_CTZ(gone);
        gone &= gone - 1u;
        t.unserved += energy[(size_t)(32 * w + bit) * io.E];
      }
    }
  }
  return t;
}

// EVENV: the kernel variant that carries the per-env roster path.  It lives in an instantiation of
// its own (like the Home-Steward house): inlined into the common kernel its register pressure cost
// every scenario 15-30 % of the component kernel (C3: 61.5 -> 80.2 us, measured).
template <bool EVENV, class IO>
PGW_HD void ev_advance(const pgw_component& c, const IO& io, int e, double kwh,
                       double& p_out, double& rew) {
  const double* dp = io.dpar + c.dpar_off;
  const double mult = dp[2];
  const double* obs_high = dp + 7;
  const double* inv_high = dp + 13;
  const double t_now = io.drow[c.dtab_off], t_next = io.drow[c.dtab_off + 1];
  EvTotals t;
  if constexpr (EVENV) {
    t = (c.flags & PGW_F_EV_PER_ENV) ? ev_charge_pass_env(c, io, e, kwh) : ev_charge_pass(c, io, e, kwh);
  } else {
    t = ev_charge_pass(c, io, e, kwh);
  }
  const double unserved = t.unserved;

  const double s_consumed = mult * t.consumed;
  const double raw[6] = {t_next, mult * (double)t.active, s_consumed, mult * t.demand,
                         t.n_deficit == 0 ? 0.0 : t.deficit_sum / (double)t.n_deficit, unserved};
  const bool rs = (c.flags & PGW_F_RESCALE) != 0;
#pragma unroll
  for (int j = 0; j < 6; ++j)
    io.obs[(size_t)(c.obs_off + j) * io.E + e] =
        obs_val(io, rs ? to_scaled(raw[j], 0.0, obs_high[j], inv_high[j]) : raw[j]);
  p_out = s_consumed;                                 // kWh per step reported as kW (:255)
  const double over = fmax(0.0, s_consumed - dp[5]);  // :135-142
  rew = div_by(-dp[3] * (unserved * unserved) + -dp[4] * (over * over), dp[6], dp[19]);
}

template <bool EVENV = false, class IO>
PGW_HD void ev_step(const pgw_component& c, const IO& io, int e, double& p_out,
                    double& rew) {
  const double* dp = io.dpar + c.dpar_off;
  double a = act_in(io, c.act_off, e);
  if (c.flags & PGW_F_RESCALE) a = to_raw(a, 0.0, 1.0);
  ev_advance<EVENV>(c, io, e, (a * dp[0]) * dp[1], p_out, rew);      // :182-183
}

template <bool EVENV = false, class IO>
PGW_HD void ev_reset(const pgw_component& c, const IO& io, int e) {
  const double* dp = io.dpar + c.dpar_off;
  const int n = io.ipar[c.ipar_off];
  if (EVENV && (c.flags & PGW_F_EV_PER_ENV)) {
    // the host has written this env's window words and initial energies (pgw_set_rows); the
    // charging set starts empty (:149)
    uint32_t* mask = io.si + (size_t)c.si_off * io.E + e;
    for (int w = 0; w < io.ipar[c.ipar_off + 1]; ++w) mask[(size_t)w * io.E] = 0u;
  } else {
    const double* e0 = dp + 21 + n;
    double* energy = io.sd + (size_t)c.sd_off * io.E + e;
    for (int i = 0; i < n; ++i) energy[(size_t)i * io.E] = e0[i];
  }
  // Hidden step with action=None -> _action_space.low = 0 (:163, :178).  With
  // rescale_spaces the reference still pushes that 0 through to_raw, i.e. 0.5.
  double a = 0.0, p, r;
  if (c.flags & PGW_F_RESCALE) a = to_raw(a, 0.0, 1.0);
  ev_advance<EVENV>(c, io, e, (a * dp[0]) * dp[1], p, r);
}

// ------------------------------------------------------------------ five-zone building
// Rolled loops over zones and observation slots: the per-thread arrays they index live in
// a scratch area (shared memory on the GPU, strided by the CTA size so lanes hit distinct
// banks; a plain local array in the host build).  Keeps the kernel's code small -- the
// fully unrolled form was 140 kB of SASS and stalled on instruction-cache misses.
enum { BSCR_T = 0, BSCR_ACT = 5, BSCR_SRC = 11, BSCR_SIZE = 35 };   // T[5], act[6], src[24]
enum { U_OUTDOOR = 0, U_SOLAR = 1, U_INTERNAL = 2, U_NEIGHBOR = 3, U_COOLING = 4 };

struct BuildingPar {
  const double *A, *B, *C, *K, *mean, *Tinit, *low, *high, *inv;
  double w_energy, w_comfort;
  const int32_t *u_kind, *u_arg, *obs_src;
};

template <class IO>
PGW_HD BuildingPar building_par(const pgw_component& c, const IO& io) {
  const double* dp = io.dpar + c.dpar_off;
  const int32_t* ip = io.ipar + c.ipar_off;
  BuildingPar b;
  b.A = dp; b.B = dp + 5; b.C = dp + 25; b.K = dp + 30; b.mean = dp + 35; b.Tinit = dp + 40;
  b.w_energy = dp[45]; b.w_comfort = dp[46];
  b.low = dp + 47; b.high = dp + 47 + c.obs_dim; b.inv = dp + 47 + 2 * c.obs_dim;
  b.u_kind = ip; b.u_arg = ip + 20; b.obs_src = ip + 40;
  return b;
}

// One selected model input of zone z (build_u_vector, dynamics.py:12-41; the host resolved
// the model's input_sel_list / neighbors into a kind + argument per input).
PGW_HD double building_input(const BuildingPar& b, const Scratch& scr, int z, int j, double t_oa,
                             const double* q_solar, const double* q_x, bool at_reset) {
  const int kind = b.u_kind[z * 4 + j];
  const double Tz = scr[BSCR_T + z];
  switch (kind) {
    case U_OUTDOOR: return t_oa - Tz;
    case U_SOLAR: return q_solar[z];
    case U_INTERNAL: return at_reset ? 0.0 : q_x[z];
    case U_NEIGHBOR: return scr[BSCR_T + b.u_arg[z * 4 + j]] - Tz;
    default:  // U_COOLING: q_cool at reset, m_dot (T_discharge - T_z) afterwards
      return at_reset ? q_x[z] : scr[BSCR_ACT + z] * (scr[BSCR_ACT + 5] - Tz);
  }
}

// state_update (dynamics.py:44-55); B already rounded through float32 on the host
PGW_HD double building_x_next(const BuildingPar& b, int z, double x, double u0, double u1,
                              double u2, double u3) {
  const double* B = b.B + z * 4;
  return b.A[z] * x + (((B[0] * u0 + B[1] * u1) + B[2] * u2) + B[3] * u3);
}

// FiveZoneROMThermalEnergyEnv.step_reward (five_zone_rom_env.py:315-335) on temps T[0..5)
PGW_HD double building_reward(const BuildingPar& b, const Scratch& scr, int t_off, double lb,
                              double ub, double p_consumed) {
  const double energy = div_by(-p_consumed, 12.0, 1.0 / 12.0);
  double comfort = 0.0;
  PGW_NO_UNROLL
  for (int z = 0; z < 5; ++z) {
    const double T = scr[t_off + z];
    const double err = fmax(fmax(T - ub, lb - T), 0.0);
    comfort += err * err;
  }
  comfort = -comfort;
  return b.w_energy * energy + b.w_comfort * comfort;
}

// get_obs (five_zone_rom_env.py:228-283): the 24 possible sources in state-dict order, then
// the selected ones (obs_src, in that same order) against the bounds in label order.
template <class IO>
PGW_HD void building_obs(const pgw_component& c, const BuildingPar& b, const IO& io,
                         int e, const Scratch& scr, double lb, double ub, double t_oa,
                         double p_consumed, double tod, bool grid) {
  PGW_NO_UNROLL
  for (int z = 0; z < 5; ++z) {
    const double T = scr[BSCR_T + z];
    scr[BSCR_SRC + z] = T;
    scr[BSCR_SRC + 5 + z] = T - ub;
    scr[BSCR_SRC + 10 + z] = lb - T;
  }
  scr[BSCR_SRC + 15] = lb;
  scr[BSCR_SRC + 16] = ub;
  scr[BSCR_SRC + 17] = t_oa;
  scr[BSCR_SRC + 18] = p_consumed;
  scr[BSCR_SRC + 19] = tod;
  if (grid) {
    scr[BSCR_SRC + 20] = io.vbus[(size_t)c.agent * io.E + e];
    scr[BSCR_SRC + 21] = io.vmin[e];
    scr[BSCR_SRC + 22] = io.vmax[e];
  }
  scr[BSCR_SRC + 23] = INFINITY;                        // p_setpoint default (:268)
  const bool rs = (c.flags & PGW_F_RESCALE) != 0;
  PGW_NO_UNROLL
  for (int slot = 0; slot < c.obs_dim; ++slot) {
    const double lo = b.low[slot], hi = b.high[slot];
    double o = clip(scr[BSCR_SRC + b.obs_src[slot]], lo, hi);   // np.clip; to_scaled's own clip
    if (rs) o = div_by(2.0 * o - (lo + hi), hi - lo, b.inv[slot]);   // is then the identity
    io.obs[(size_t)(c.obs_off + slot) * io.E + e] = obs_val(io, o);
  }
}

template <class IO>
PGW_HD void building_reset(const pgw_component& c, const IO& io, int e) {
  const BuildingPar b = building_par(c, io);
  const Scratch& scr = io.scr;
  const double* row = io.drow + c.dtab_off;
  double* sd = io.sd + (size_t)c.sd_off * io.E + e;
  for (int z = 0; z < 5; ++z) scr[BSCR_T + z] = b.Tinit[z];
  PGW_NO_UNROLL
  for (int z = 0; z < 5; ++z) {
    // the inputs are built once from T_init; two filter updates (dynamics.py:58-72)
    const double u0 = building_input(b, scr, z, 0, row[0], row + 1, row + 6, true);
    const double u1 = building_input(b, scr, z, 1, row[0], row + 1, row + 6, true);
    const double u2 = building_input(b, scr, z, 2, row[0], row + 1, row + 6, true);
    const double u3 = building_input(b, scr, z, 3, row[0], row + 1, row + 6, true);
    double x = sd[(size_t)z * io.E];                    // x persists across resets (:94)
    for (int rep = 0; rep < 2; ++rep) {
      x = building_x_next(b, z, x, u0, u1, u2, u3);
      x += b.K[z] * ((b.Tinit[z] - b.mean[z]) - b.C[z] * x);
    }
    sd[(size_t)z * io.E] = x;
    scr[BSCR_ACT + z] = b.C[z] * x + b.mean[z];         // new temps, parked until all zones are done
  }
  for (int z = 0; z < 5; ++z) scr[BSCR_T + z] = scr[BSCR_ACT + z];
  sd[(size_t)5 * io.E] = 0.0;                           // p_consumed
  building_obs(c, b, io, e, scr, row[12], row[13], row[11], 0.0, row[14],
               (c.flags & PGW_F_GRID_AWARE) != 0);
}

template <class IO>
PGW_HD void building_step(const pgw_component& c, const IO& io, int e, double& p_out,
                          double& rew) {
  const BuildingPar b = building_par(c, io);
  const Scratch& scr = io.scr;
  const double* row = io.drow + c.dtab_off;
  double* sd = io.sd + (size_t)c.sd_off * io.E + e;
  const bool rs = (c.flags & PGW_F_RESCALE) != 0;
  double flow = 0.0;
  PGW_NO_UNROLL
  for (int i = 0; i < 6; ++i) {                         // action bounds :22-26
    const double lo = i < 4 ? 0.22 : (i == 4 ? 0.32 : 10.0);
    const double hi = i < 4 ? 2.2 : (i == 4 ? 3.2 : 16.0);
    const double a = act_in(io, c.act_off + i, e);
    const double raw = rs ? to_raw(a, lo, hi) : a;
    scr[BSCR_ACT + i] = raw;
    if (i < 5) flow = i == 0 ? raw : flow + raw;
  }
  for (int z = 0; z < 5; ++z) scr[BSCR_T + z] = b.C[z] * sd[(size_t)z * io.E] + b.mean[z];
  if (c.flags & PGW_F_STALE_REWARD)                     // stand-alone agent: pre-step state (:215)
    rew = building_reward(b, scr, BSCR_T, row[15], row[16], sd[(size_t)5 * io.E]);
  const double t_oa = row[0], t_dis = scr[BSCR_ACT + 5];
  PGW_NO_UNROLL
  for (int z = 0; z < 5; ++z) {                         // all inputs use the OLD temperatures
    const double u0 = building_input(b, scr, z, 0, t_oa, row + 1, row + 6, false);
    const double u1 = building_input(b, scr, z, 1, t_oa, row + 1, row + 6, false);
    const double u2 = building_input(b, scr, z, 2, t_oa, row + 1, row + 6, false);
    const double u3 = building_input(b, scr, z, 3, t_oa, row + 1, row + 6, false);
    const double x = building_x_next(b, z, sd[(size_t)z * io.E], u0, u1, u2, u3);
    sd[(size_t)z * io.E] = x;
    scr[BSCR_SRC + z] = b.C[z] * x + b.mean[z];         // new temps, parked in the source area
  }
  for (int z = 0; z < 5; ++z) scr[BSCR_T + z] = scr[BSCR_SRC + z];
  // flow**3: the reference calls libm pow; x*x*x differs from it by at most 1 ulp
  const double p = (0.0076 * ((flow * flow) * flow) + 4.8865) + fmax(0.0, flow * (t_oa - t_dis));
  sd[(size_t)5 * io.E] = p;
  building_obs(c, b, io, e, scr, row[12], row[13], row[11], p, row[14],
               (c.flags & PGW_F_GRID_AWARE) != 0);
  if (!(c.flags & PGW_F_STALE_REWARD)) rew = building_reward(b, scr, BSCR_T, row[12], row[13], p);
  p_out = p;
}

// ---- fast path: the reference's shipped model + default observation set ----------------
// PGW_F_BUILDING_FAST is set by the host when (a) every zone's model inputs are
// [outdoor, cooling, neighbour, solar] (the input_sel_list of state_space_model.p) and
// (b) the observation set is defaults.obs_config (upper/lower violation per zone, comfort
// band, outdoor temperature, p_consumed, time of day).  Same arithmetic, same order of
// operations as the generic path, but straight-line code on registers: the table-driven
// form spends ~85 % of its instructions on indexing rather than on float64 math.
PGW_HD double pick5(const double T[5], int i) {
  double v = T[0];
  v = i == 1 ? T[1] : v;
  v = i == 2 ? T[2] : v;
  v = i == 3 ? T[3] : v;
  v = i == 4 ? T[4] : v;
  return v;
}

template <class IO>
PGW_HD void building_step_fast(const pgw_component& c, const IO& io, int e, double& p_out,
                               double& rew) {
  const double* dp = io.dpar + c.dpar_off;
  const int32_t* u_arg = io.ipar + c.ipar_off + 20;
  const double *A = dp, *B = dp + 5, *C = dp + 25, *mean = dp + 35;
  const double *low = dp + 47, *high = dp + 62, *inv = dp + 77;     // obs_dim == 15
  const double* row = io.drow + c.dtab_off;
  const size_t E = (size_t)io.E;
  const bool rs = (c.flags & PGW_F_RESCALE) != 0;
  const double kLow[6] = {0.22, 0.22, 0.22, 0.22, 0.32, 10.0};      // action bounds :22-26
  const double kHigh[6] = {2.2, 2.2, 2.2, 2.2, 3.2, 16.0};

  double* sp = io.sd + (size_t)c.sd_off * E + e;
  double act[6], x[5], T[5], Tn[5];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const double a = act_in(io, c.act_off + i, e);
    act[i] = rs ? to_raw(a, kLow[i], kHigh[i]) : a;
  }
#pragma unroll
  for (int z = 0; z < 5; ++z) {
    x[z] = sp[z * E];
    T[z] = C[z] * x[z] + mean[z];
  }
  const double t_oa = row[0], t_dis = act[5];
#pragma unroll
  for (int z = 0; z < 5; ++z) {                  // inputs [outdoor, cooling, neighbour, solar]
    const double u0 = t_oa - T[z];
    const double u1 = act[z] * (t_dis - T[z]);
    const double u2 = pick5(T, u_arg[z * 4 + 2]) - T[z];
    const double u3 = row[1 + z];
    const double* Bz = B + z * 4;
    const double xn = A[z] * x[z] + (((Bz[0] * u0 + Bz[1] * u1) + Bz[2] * u2) + Bz[3] * u3);
    sp[z * E] = xn;
    Tn[z] = C[z] * xn + mean[z];
  }
  const double flow = (((act[0] + act[1]) + act[2]) + act[3]) + act[4];
  const double p = (0.0076 * ((flow * flow) * flow) + 4.8865) + fmax(0.0, flow * (t_oa - t_dis));
  sp[5 * E] = p;

  const double lb = row[12], ub = row[13];
  auto* op = io.obs + (size_t)c.obs_off * E + e;
  double comfort = 0.0;
#pragma unroll
  for (int z = 0; z < 5; ++z) {
    const double up = Tn[z] - ub, lo = lb - Tn[z];
    double o = clip(up, low[z], high[z]);
    op[z * E] = obs_val(io, rs ? div_by(2.0 * o - (low[z] + high[z]), high[z] - low[z], inv[z]) : o);
    o = clip(lo, low[5 + z], high[5 + z]);
    op[(5 + z) * E] = obs_val(
        io, rs ? div_by(2.0 * o - (low[5 + z] + high[5 + z]), high[5 + z] - low[5 + z], inv[5 + z]) : o);
    const double err = fmax(fmax(up, lo), 0.0);
    comfort += err * err;
  }
  const double tail[5] = {lb, ub, row[11], p, row[14]};
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const int s = 10 + j;
    const double o = clip(tail[j], low[s], high[s]);
    op[s * E] = obs_val(io, rs ? div_by(2.0 * o - (low[s] + high[s]), high[s] - low[s], inv[s]) : o);
  }
  const double energy = div_by(-p, 12.0, 1.0 / 12.0);
  rew = dp[45] * energy + dp[46] * (-comfort);
  p_out = p;
}

// ------------------------------------------------------------------ Home-Steward house
// gridworld/base_hs.py:12-199 + agents/*/*_hs.py: the components of a house are stepped in
// order and share the step's available solar / battery / grid power through a "meta state"
// that also survives from step to step.  On the device that state is a small per-thread record
// loaded by the leading HS_BEGIN pseudo-component and stored at the end of the house's step.
// Divisions by per-env quantities (the blended costs) are plain IEEE float64 divisions; divisions
// by constants use the host-computed reciprocal + FMA correction of div_by (same quotient).
struct HsMeta {
  double pv_power, es_power, grid_power, pv_cost, es_cost, grid_cost;
  double r[PGW_HS_MAX_COMPONENTS];        // per-component reward terms, summed in order at the end
  double es_pen[PGW_HS_MAX_COMPONENTS];   // storage: pending penalty (needs the FINAL meta), or 0
  int n;
};

// Optional per-component telemetry (PGW_F_TELEMETRY): the numbers of the reference's
// ``step_meta`` records, kPgwTelRows state rows behind the component's own state:
//   0 cost, 1 reward (as evaluated inside the component's step), 2 raw action,
//   3 solar / 4 battery / 5 grid power consumed, 6.. device_custom_info entries
struct HsTel {
  double* p;
  int E;
  PGW_HD void put(int r, double v) const { if (p) p[(size_t)r * E] = v; }
};
template <bool TEL, class IO>
PGW_HD HsTel hs_tel(const pgw_component& c, const IO& io, int e, int own_rows) {
  HsTel t;
  t.E = io.E;
  t.p = (TEL && (c.flags & PGW_F_TELEMETRY)) ? io.sd + (size_t)(c.sd_off + own_rows) * io.E + e
                                             : nullptr;
  return t;
}

// HS_BEGIN  dpar: max_grid_power   dtab: grid_cost of the event
//           state: pv_power, es_power, es_cost, pv_cost, grid_power (5 rows, the meta state)
template <class IO>
PGW_HD void hs_begin(const pgw_component& c, const IO& io, int e, HsMeta& m, bool first_reset) {
  double* sd = io.sd + (size_t)c.sd_off * io.E + e;
  if (first_reset) {                                   // base_hs.py:53-61
    for (int r = 0; r < 5; ++r) sd[(size_t)r * io.E] = 0.0;
  }
  m.pv_power = sd[0];
  m.es_power = sd[(size_t)1 * io.E];
  m.es_cost = sd[(size_t)2 * io.E];
  m.pv_cost = sd[(size_t)3 * io.E];
  m.grid_power = io.dpar[c.dpar_off];                  // :125
  m.grid_cost = io.drow[c.dtab_off];                   // :124
  m.n = 0;
}

template <class IO>
PGW_HD void hs_end(const pgw_component& c, const IO& io, int e, const HsMeta& m, bool store,
                   double& r_agent) {
  if (store) {
    double* sd = io.sd + (size_t)c.sd_off * io.E + e;  // c = the HS_BEGIN descriptor
    sd[0] = m.pv_power;
    sd[(size_t)1 * io.E] = m.es_power;
    sd[(size_t)2 * io.E] = m.es_cost;
    sd[(size_t)3 * io.E] = m.pv_cost;
    sd[(size_t)4 * io.E] = m.grid_power;
  }
  // step_reward(**meta_state) after every component has stepped (base_hs.py:176, :184-199)
  double r = 0.0;
  const bool pen = m.pv_power > 0.0 && m.es_power > 0.0;     // energy_storage_env_hs.py:176-181
  for (int i = 0; i < m.n; ++i) {
    double ri = m.r[i];
    if (pen && m.es_pen[i] != 0.0) ri -= m.es_pen[i];
    r += ri;
  }
  r_agent = r;
}

// HS_PV  dpar: obs_low, obs_high, 1/(high-low)   dtab: scaled profile value of the event
template <bool TEL, class IO>
PGW_HD void hs_pv_step(const pgw_component& c, const IO& io, int e, HsMeta& m, bool reset,
                       double& p_out) {
  const double* dp = io.dpar + c.dpar_off;
  const bool rs = (c.flags & PGW_F_RESCALE) != 0;
  const double data = io.drow[c.dtab_off];
  const double raw = -data;                            // pv_profile_env_hs.py:110
  io.obs[(size_t)c.obs_off * io.E + e] = obs_val(io, rs ? to_scaled(raw, dp[0], dp[1], dp[2]) : raw);
  if (reset) {
    m.pv_power = -raw;                                 // only the reset chain sees it (:121-124)
    p_out = 0.0;
    return;
  }
  double a = act_in(io, c.act_off, e);
  if (rs) a = to_raw(a, 0.98, 1.0);                    // :100-101, :140-141
  const double p = a * (-raw);                         // :149
  m.pv_power = p;                                      // :153
  m.r[m.n] = 0.0; m.es_pen[m.n] = 0.0; ++m.n;
  const HsTel t = hs_tel<TEL>(c, io, e, 0);                 // :154-158
  t.put(0, 0.0); t.put(1, 0.0); t.put(2, a); t.put(3, -raw); t.put(4, 0.0); t.put(5, 0.0);
  t.put(6, -raw); t.put(7, p);
  p_out = p;
}

// HS_STORAGE  dpar: lo, hi, eta_c, eta_d, max_power, dt_hours, initial mean, initial cost,
//                   max_storage_cost, 1/(hi-lo), 1/max_storage_cost, 1/eta_d, 1/dt, 1/eta_c
//             ipar: storage ordinal
//             state: SOC, current_cost
template <class IO>
PGW_HD void hs_storage_obs(const pgw_component& c, const IO& io, int e, double soc, double cost) {
  const double* dp = io.dpar + c.dpar_off;
  const bool rs = (c.flags & PGW_F_RESCALE) != 0;
  io.obs[(size_t)c.obs_off * io.E + e] = obs_val(io, rs ? to_scaled(soc, dp[0], dp[1], dp[9]) : soc);
  io.obs[(size_t)(c.obs_off + 1) * io.E + e] = obs_val(io, rs ? to_scaled(cost, 0.0, dp[8], dp[10]) : cost);
}

template <class IO>
PGW_HD void hs_storage_reset(const pgw_component& c, const IO& io, int e, bool first_reset) {
  const double* dp = io.dpar + c.dpar_off;
  double* sd = io.sd + (size_t)c.sd_off * io.E + e;
  const int ord = io.ipar[c.ipar_off];
  const double init = io.init_soc != nullptr ? io.init_soc[(size_t)ord * io.E + e] : dp[6];
  // energy_storage_env_hs.py:84-96: a drawn SOC is used as is, an explicit one is clipped
  const double soc = (io.init_soc != nullptr && !io.clip_init_soc) ? init : clip(init, dp[0], dp[1]);
  sd[0] = soc;
  if (first_reset) sd[(size_t)1 * io.E] = dp[7];       // current_cost is never reset (:39)
  hs_storage_obs(c, io, e, soc, sd[(size_t)1 * io.E]);
}

template <bool TEL, class IO>
PGW_HD void hs_storage_step(const pgw_component& c, const IO& io, int e, HsMeta& m,
                            double& p_out) {
  const double* dp = io.dpar + c.dpar_off;
  const double lo = dp[0], hi = dp[1], eta_c = dp[2], eta_d = dp[3], pmax = dp[4], dt = dp[5];
  double* sd = io.sd + (size_t)c.sd_off * io.E + e;
  double soc = sd[0], cost = sd[(size_t)1 * io.E];
  double a = act_in(io, c.act_off, e);
  if (c.flags & PGW_F_RESCALE) a = to_raw(a, -1.0, 1.0);
  double power = a * pmax;
  // validate_power :111-143
  const double inv_eta_d = dp[11], inv_dt = dp[12], inv_eta_c = dp[13];
  if (power > 0.0) {
    const double delta = div_by(power * dt, eta_d, inv_eta_d);
    if (soc <= lo) power = 0.0;
    else if (soc - delta < lo) power = div_by(soc - lo, dt, inv_dt) * eta_d;
  } else if (power < 0.0) {
    const double delta = -(power * dt * eta_c);
    if (soc >= hi) power = 0.0;
    else if (soc + delta > hi) power = -div_by(div_by(hi - soc, dt, inv_dt), eta_c, inv_eta_c);
  }
  double delta_cost = 0.0, solar_taken = 0.0, grid_taken = 0.0;
  const double solar_cap = m.pv_power, grid_cap = m.grid_power;
  if (power == 0.0) {                                  // :215-217
    m.es_power = 0.0;
  } else if (power < 0.0) {                            // charging :219-245
    const double delta_storage = eta_c * power * dt;
    const double solar_used = fmin(-power, m.pv_power);
    const double grid_used = fmin(m.grid_power, -power - solar_used);
    delta_cost = (m.pv_cost * solar_used + m.grid_cost * grid_used) / (solar_used + grid_used);
    cost = (soc * cost - delta_storage * delta_cost) / (soc - delta_storage);
    soc -= delta_storage;
    soc = fmin(soc, hi);
    m.pv_power = fmax(0.0, m.pv_power - solar_used);
    m.grid_power = fmax(0.0, m.grid_power - grid_used);
    m.es_power = 0.0;
    solar_taken = solar_used;
    grid_taken = grid_used;
  } else {                                             // discharging :248-253
    const double delta_storage = div_by(power * dt, eta_d, inv_eta_d);
    soc = fmax(soc - delta_storage, lo);
    m.es_power = power;
  }
  m.es_cost = 0.0;                                     // :256
  sd[0] = soc;
  sd[(size_t)1 * io.E] = cost;
  hs_storage_obs(c, io, e, soc, cost);
  const double real_power = -power;                    // :258
  // step_reward :161-190; the solar-available penalty is decided on the final meta (hs_end)
  double step_cost = 0.0;
  if (!(real_power < 0.0)) step_cost = delta_cost * eta_c * real_power * dt;
  const double smax = fmax(lo, hi);
  m.r[m.n] = -step_cost;
  m.es_pen[m.n] = soc < smax ? dp[8] * (smax - soc) : 0.0;
  const HsTel t = hs_tel<TEL>(c, io, e, 2);                 // :262-271
  if (t.p) {
    double rew = -step_cost;                           // reward as seen inside the step (:264)
    if (m.pv_power > 0.0 && m.es_power > 0.0 && m.es_pen[m.n] != 0.0) rew -= m.es_pen[m.n];
    t.put(0, step_cost); t.put(1, rew); t.put(2, a);
    t.put(3, solar_taken); t.put(4, 0.0); t.put(5, grid_taken);
    t.put(6, soc); t.put(7, power); t.put(8, solar_cap - solar_taken);
    t.put(9, grid_cap - grid_taken); t.put(10, m.es_power);
  }
  ++m.n;
  p_out = real_power;
}

// HS_EV  dpar: as the stock station up to e0[n], then max_charge_cost, 60 / minutes_per_step,
//              1 / max_charge_cost
//        dtab: evaluation time, new time      itab: as the stock station
//        state: n energy rows + current_cost; words of the charging set
template <bool TEL, class IO>
PGW_HD void hs_ev_advance(const pgw_component& c, const IO& io, int e, double a_raw, HsMeta& m,
                          bool reset, double& p_out) {
  const double* dp = io.dpar + c.dpar_off;
  const int n = io.ipar[c.ipar_off];
  const double mult = dp[2];
  const double* obs_high = dp + 7;
  const double max_cost = dp[21 + 2 * n], per_hour = dp[22 + 2 * n];
  const double t_eval = io.drow[c.dtab_off], t_new = io.drow[c.dtab_off + 1];
  double* cost_p = io.sd + (size_t)(c.sd_off + n) * io.E + e;
  const double kwh = (a_raw * dp[0]) * dp[1];          // ev_charging_env_hs.py:203-204
  const HsTel tel = hs_tel<TEL>(c, io, e, n + 1);
  const int words = io.ipar[c.ipar_off + 1];
  uint32_t* mask = io.si + (size_t)c.si_off * io.E + e;
  uint32_t old_mask[4] = {0u, 0u, 0u, 0u};             // telemetry: vehicles that stop charging
  if (tel.p && !reset)
    for (int w = 0; w < words && w < 4; ++w) old_mask[w] = mask[(size_t)w * io.E];
  const EvTotals t = ev_charge_pass(c, io, e, kwh);
  const double real_power = mult * t.consumed;         // :281
  const double power = real_power * per_hour;          // :285
  double cost = *cost_p;                               // kept across episodes, 0 at creation
  HsMeta loc = m;                                      // the hidden step of reset discards these
  const double cap_pv = m.pv_power, cap_es = m.es_power, cap_grid = m.grid_power;
  double solar_used = 0.0, battery_used = 0.0, grid_used = 0.0;
  if (power == 0.0 || a_raw == 0.0) {                  // :292-293
    cost = 0.0;
  } else {
    solar_used = fmin(power, loc.pv_power);
    if (loc.es_cost < loc.grid_cost) {                 // :304-309
      battery_used = fmin(loc.es_power, power - solar_used);
      grid_used = fmin(loc.grid_power, power - solar_used - battery_used);
    } else {
      grid_used = fmin(loc.grid_power, power - solar_used);
      battery_used = fmin(loc.es_power, power - solar_used - grid_used);
    }
    if (solar_used + grid_used + battery_used > 0.0)
      cost = (loc.pv_cost * solar_used + loc.grid_cost * grid_used + loc.es_cost * battery_used) /
             (solar_used + grid_used + battery_used);
    loc.pv_power = fmax(0.0, loc.pv_power - solar_used);
    loc.es_power = fmax(0.0, loc.es_power - battery_used);
    loc.grid_power = fmax(0.0, loc.grid_power - grid_used);
  }
  *cost_p = cost;
  const double raw[7] = {t_new, mult * (double)t.active, real_power, mult * t.demand,
                         t.n_deficit == 0 ? 0.0 : t.deficit_sum / (double)t.n_deficit, t.unserved,
                         cost};
  const bool rs = (c.flags & PGW_F_RESCALE) != 0;
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    const double hi = j < 6 ? obs_high[j] : max_cost;
    const double inv = j < 6 ? dp[13 + j] : dp[23 + 2 * n];
    io.obs[(size_t)(c.obs_off + j) * io.E + e] = obs_val(io, rs ? to_scaled(raw[j], 0.0, hi, inv) : raw[j]);
  }
  if (!reset) {
    m.pv_power = loc.pv_power; m.es_power = loc.es_power; m.grid_power = loc.grid_power;
    // :178-191
    const double step_cost = cost * real_power;
    m.r[m.n] = -(step_cost + dp[3] * (t.unserved * t.unserved));
    m.es_pen[m.n] = 0.0;
    if (tel.p) {                                       // :318-323
      int departed = 0;
      for (int w = 0; w < words && w < 4; ++w)
        departed += PGW_POPC(old_mask[w] & ~mask[(size_t)w * io.E]);
      tel.put(0, step_cost); tel.put(1, m.r[m.n]); tel.put(2, a_raw);
      tel.put(3, solar_used); tel.put(4, battery_used); tel.put(5, grid_used);
      tel.put(6, power); tel.put(7, t.unserved); tel.put(8, (double)t.active);
      tel.put(9, (double)departed); tel.put(10, cap_pv - solar_used);
      tel.put(11, cap_es - battery_used); tel.put(12, cap_grid - grid_used);
    }
    ++m.n;
  }
  p_out = real_power;
}

template <bool TEL, class IO>
PGW_HD void hs_ev_reset(const pgw_component& c, const IO& io, int e, HsMeta& m) {
  const double* dp = io.dpar + c.dpar_off;
  const int n = io.ipar[c.ipar_off];
  const double* e0 = dp + 21 + n;
  double* energy = io.sd + (size_t)c.sd_off * io.E + e;
  for (int i = 0; i < n; ++i) energy[(size_t)i * io.E] = e0[i];
  double a = 0.0, p;                                   // hidden step, action = space low (:151, :199)
  if (c.flags & PGW_F_RESCALE) a = to_raw(a, 0.0, 1.0);
  hs_ev_advance<TEL>(c, io, e, a, m, true, p);
}

// HS_DEVICES  dpar: minutes_per_step / 60, obs_high[k], 1/obs_high[k]     ipar: k (columns)
//             dtab: scaled row [k] (observation), unscaled row [k] (demand)
template <bool TEL, class IO>
PGW_HD void hs_devices_step(const pgw_component& c, const IO& io, int e, HsMeta& m, bool reset,
                            double& p_out) {
  const double* dp = io.dpar + c.dpar_off;
  const int k = io.ipar[c.ipar_off];
  const bool rs = (c.flags & PGW_F_RESCALE) != 0;
  const double* row = io.drow + c.dtab_off;
  for (int j = 0; j < k; ++j)
    io.obs[(size_t)(c.obs_off + j) * io.E + e] =
        obs_val(io, rs ? to_scaled(row[j], 0.0, dp[1 + j], dp[1 + k + j]) : row[j]);
  p_out = 0.0;
  if (reset) return;
  double a = act_in(io, c.act_off, e);
  if (rs) a = to_raw(a, 0.99, 1.0);                    // devices_env_hs.py:98-99
  double total = 0.0;
  for (int j = 0; j < k; ++j) total += row[k + j];     // :165
  const double p = a * total;
  double cost = 0.0, solar_used = 0.0, battery_used = 0.0, grid_used = 0.0;
  if (rint(p * 1000.0) != 0.0) {                       // round(p, 3) == 0.0 (:174)
    solar_used = fmin(p, m.pv_power);
    battery_used = fmin(m.es_power, p - solar_used);
    grid_used = fmin(m.grid_power, p - solar_used - battery_used);
    cost = (m.pv_cost * solar_used + m.grid_cost * grid_used + m.es_cost * battery_used) /
           (solar_used + grid_used + battery_used);
    // the reference hands back the meta it copied BEFORE this allocation (:163, :201):
    // what the devices consume never reaches the meta state
  }
  const double step_cost = cost * p * dp[0];           // :128-131
  m.r[m.n] = -step_cost;
  m.es_pen[m.n] = 0.0;
  ++m.n;
  const HsTel t = hs_tel<TEL>(c, io, e, 0);                 // :194-198
  t.put(0, step_cost); t.put(1, -step_cost); t.put(2, a);
  t.put(3, solar_used); t.put(4, battery_used); t.put(5, grid_used);
  t.put(6, p); t.put(7, m.pv_power - solar_used); t.put(8, m.es_power - battery_used);
  t.put(9, m.grid_power - grid_used);
  p_out = p;
}

// ------------------------------------------------------------------ one agent of one env
// MultiComponentEnv.step (base.py:114-139): components in order, real power summed,
// reward = sum of the components' post-step rewards.  A single-component agent is the
// one-element case (its own step reward, multiagent_env.py:168).
PGW_HD bool is_house(const pgw_agent& ag, const pgw_component* comps) {
  return comps[ag.comp_begin].type == PGW_HS_BEGIN;
}

// Home-Steward house (base_hs.py:120-178).  Kept apart from agent_step so that kernels of
// scenarios without a house do not carry its code and stack frame.
template <bool TEL, class IO>
PGW_HD void house_step(const pgw_agent& ag, const pgw_component* comps, const IO& io, int e,
                       double& p_agent, double& r_agent) {
  p_agent = 0.0;
  HsMeta m;
  hs_begin(comps[ag.comp_begin], io, e, m, false);
  for (int ci = ag.comp_begin + 1; ci < ag.comp_end; ++ci) {
    const pgw_component c = comps[ci];
    double p = 0.0;
    switch (c.type) {
      case PGW_HS_PV: hs_pv_step<TEL>(c, io, e, m, false, p); break;
      case PGW_HS_STORAGE: hs_storage_step<TEL>(c, io, e, m, p); break;
      case PGW_HS_EV: {
        double a = act_in(io, c.act_off, e);
        if (c.flags & PGW_F_RESCALE) a = to_raw(a, 0.0, 1.0);
        hs_ev_advance<TEL>(c, io, e, a, m, false, p);
        break;
      }
      case PGW_HS_DEVICES: hs_devices_step<TEL>(c, io, e, m, false, p); break;
      default: break;
    }
    p_agent += p;
  }
  hs_end(comps[ag.comp_begin], io, e, m, true, r_agent);
}

// base_hs.py:67-92; the meta state itself is not reset
template <bool TEL, class IO>
PGW_HD void house_reset(const pgw_agent& ag, const pgw_component* comps, const IO& io, int e,
                        bool first_reset) {
  HsMeta m;
  hs_begin(comps[ag.comp_begin], io, e, m, first_reset);
  for (int ci = ag.comp_begin + 1; ci < ag.comp_end; ++ci) {
    const pgw_component c = comps[ci];
    double p;
    switch (c.type) {
      case PGW_HS_PV: hs_pv_step<TEL>(c, io, e, m, true, p); break;
      case PGW_HS_STORAGE: hs_storage_reset(c, io, e, first_reset); break;
      case PGW_HS_EV: hs_ev_reset<TEL>(c, io, e, m); break;
      case PGW_HS_DEVICES: hs_devices_step<TEL>(c, io, e, m, true, p); break;
      default: break;
    }
  }
}

template <bool EVENV = false, class IO>
PGW_HD void agent_step(const pgw_agent& ag, const pgw_component* comps, const IO& io, int e,
                       double& p_agent, double& r_agent) {
  p_agent = 0.0;
  r_agent = 0.0;
  for (int ci = ag.comp_begin; ci < ag.comp_end; ++ci) {
    const pgw_component c = comps[ci];
    double p = 0.0, r = 0.0;
    switch (c.type) {
      case PGW_STORAGE: storage_step(c, io, e, p); break;
      case PGW_PV: pv_step(c, io, e, p, r); break;
      case PGW_EV: ev_step<EVENV>(c, io, e, p, r); break;
      case PGW_BUILDING:
        if (c.flags & PGW_F_BUILDING_FAST) building_step_fast(c, io, e, p, r);
        else building_step(c, io, e, p, r);
        break;
      default: break;
    }
    p_agent += p;
    r_agent += r;
  }
}

template <bool EVENV = false, class IO>
PGW_HD void agent_reset(const pgw_agent& ag, const pgw_component* comps, const IO& io, int e) {
  for (int ci = ag.comp_begin; ci < ag.comp_end; ++ci) {
    const pgw_component c = comps[ci];
    switch (c.type) {
      case PGW_STORAGE: storage_reset(c, io, e); break;
      case PGW_PV: pv_obs(c, io, e, -io.drow[c.dtab_off]); break;
      case PGW_EV: ev_reset<EVENV>(c, io, e); break;
      case PGW_BUILDING: building_reset(c, io, e); break;
      default: break;
    }
  }
}

}  // namespace pgw
