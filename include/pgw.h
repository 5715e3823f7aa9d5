/*
 * pgw.h -- C ABI of the B200 batched simulator for PowerGridworld's
 * MultiAgentEnv.step hot path.
 *
 * The reference (lmchion/PowerGridworld) has no FFI of its own: its boundary is
 * three Python protocols chosen by class objects inside config dicts.  This ABI
 * is what sits underneath those protocols here; each entry point names the
 * reference interface it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - Every per-env array is "rows x E" with the env index fastest varying
 *     (structure of arrays): element (row, e) lives at  ptr[row * E + e].
 *   - All floating point is IEEE double (the reference computes in float64); the *_f32
 *     entry points take float actions and observations instead (computed in double).
 *   - Buffers passed to pgw_reset / pgw_step / pgw_get are DEVICE pointers owned
 *     by the caller (e.g. torch tensors); the *_host variants take HOST pointers
 *     and perform the copies themselves.
 *   - Functions return 0 on success, a negative pgw_status otherwise; the text of
 *     the last error of the calling thread is available from pgw_last_error().
 *     Nothing throws across the ABI.  Power-flow non-convergence is data
 *     (PGW_FIELD_PF_ITERS / pgw_stats), not an error.
 *   - Calls on one handle are stream ordered and not re-entrant.
 *   - All envs of a handle advance in lock step (episode termination in the
 *     reference is a pure function of the step count, see SURVEY.md 3.1-6), so
 *     the episode clock is a scalar that lives on the device.
 */
#ifndef PGW_H_
#define PGW_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGW_ABI_VERSION 1

typedef enum pgw_status {
  PGW_OK = 0,
  PGW_ERR_INVALID = -1,   /* malformed spec / argument */
  PGW_ERR_CUDA = -2,      /* CUDA runtime error (text in pgw_last_error) */
  PGW_ERR_ARCH = -3,      /* device is not sm_100 */
  PGW_ERR_STATE = -4,     /* step before reset, or step past the end of the episode */
  PGW_ERR_NOMEM = -5
} pgw_status;

/* Component kinds = the reference's ComponentEnv subclasses on the hot path. */
typedef enum pgw_component_type {
  PGW_STORAGE = 1,   /* gridworld/agents/energy_storage/energy_storage_env.py:11-181 */
  PGW_PV = 2,        /* gridworld/agents/pv/pv_profile_env.py:15-148               */
  PGW_EV = 3,        /* gridworld/agents/vehicles/ev_charging_env.py:17-275        */
  PGW_BUILDING = 4,  /* gridworld/agents/buildings/five_zone_rom_env.py:60-335     */
  /* Home-Steward house (gridworld/base_hs.py:12-199): an agent whose FIRST component is
   * PGW_HS_BEGIN is stepped as an HSMultiComponentEnv -- its components share the step's
   * available solar / battery / grid power and the composite reward is evaluated on the
   * final meta state. */
  PGW_HS_BEGIN = 5,    /* pseudo component: meta state + grid cost (no action, no observation) */
  PGW_HS_PV = 6,       /* gridworld/agents/pv/pv_profile_env_hs.py:15-169                  */
  PGW_HS_STORAGE = 7,  /* gridworld/agents/energy_storage/energy_storage_env_hs.py:10-273  */
  PGW_HS_EV = 8,       /* gridworld/agents/vehicles/ev_charging_env_hs.py:15-336           */
  PGW_HS_DEVICES = 9   /* gridworld/agents/devices/devices_env_hs.py:14-205                */
} pgw_component_type;

/* pgw_component.flags */
#define PGW_F_RESCALE 1u        /* rescale_spaces=True: actions/obs in [-1, 1] (gridworld/utils.py:9-43) */
#define PGW_F_GRID_AWARE 2u     /* PVEnv(grid_aware=True): min_voltage appended to the obs; building:
                                   some bus/min/max_voltage entry is observed                          */
#define PGW_F_PV_VOLT_REWARD 4u /* ThisPVEnv.step_reward, gridworld/scenarios/heterogeneous.py:46-52   */
#define PGW_F_BUILDING_FAST 16u /* building with the shipped model's input pattern and the default
                                   15-entry observation set: straight-line register code path   */
#define PGW_F_TELEMETRY 32u     /* Home-Steward component: PGW_HS_TEL_ROWS extra double state rows behind
                                   its own state receive the numbers of the reference's step_meta record
                                   (cost, reward, raw action, solar / battery / grid power consumed,
                                   device_custom_info entries)                                         */
#define PGW_HS_TEL_ROWS 13
#define PGW_F_EV_PER_ENV 64u    /* EVChargingEnv(randomize=True) in a batch: every env instance parks its OWN
                                   roster sample (ev_charging_env.py:154-157).  ipar = n, ceil(n/32), 0; the
                                   station's uint32 state is ceil(n/32) charging-set words followed by n
                                   window words (floor(start) << 16 | floor(end), minutes) per env; the
                                   window words and the n initial energies are written by the host with
                                   pgw_set_rows before every pgw_reset; event row = {t, t_next} only        */
#define PGW_F_STALE_REWARD 8u   /* stand-alone building agent: reward from the pre-step state
                                   (five_zone_rom_env.py:215 precedes :223)                            */

/*
 * One component instance of the scenario (identical for every env).
 * Parameter blocks live in pgw_spec.dpar / ipar at dpar_off / ipar_off:
 *
 *  (entries named 1/x hold the correctly rounded reciprocal, computed on the host, used
 *   by the kernels' division-by-constant: multiply + one FMA correction = IEEE quotient)
 *  STORAGE  dpar: lo, hi, eta_charge, eta_discharge, max_power, dt_hours, initial mean,
 *                 1/(hi-lo), 1/eta_discharge, 1/dt_hours
 *           ipar: storage ordinal (row of init_soc)
 *           state: 1 double row (SOC)                      action 1, obs 1
 *  PV       dpar: obs_low0, obs_high0, obs_low1, obs_high1, 1/(high0-low0), 1/(high1-low1)
 *           dtab: profile value of the event              action 1, obs 1 (+1 grid aware)
 *  EV       dpar: rate_kw, step_hours, multiplier, unserved_penalty, peak_penalty,
 *                 peak_threshold, reward_scale, obs_high[6], 1/obs_high[6], 1/reward_scale,
 *                 1/60, end_park_min[n], e0_kwh[n]
 *           ipar: n, words(=ceil(n/32)), list capacity m
 *           dtab: time_now, time_next, hours_left[m], 1/hours_left[m] (per window slot)
 *           itab: n_window, n_left, window[m], left[m]
 *           state: n double rows (remaining kWh), words uint32 rows (charging set)
 *                                                          action 1, obs 6
 *  BUILDING dpar: A[5], B[20] (float32-rounded), C[5], K[5], mean[5], T_init[5],
 *                 w_energy(=alpha*0.5), w_comfort(=1-alpha), low[obs_dim], high[obs_dim],
 *                 1/(high-low)[obs_dim]
 *           ipar: u_kind[20], u_arg[20] (model input j of zone z: 0 outdoor, 1 solar,
 *                 2 internal, 3 neighbour(arg), 4 cooling), obs_src[obs_dim] (state-dict
 *                 index of each observation slot, 0..23)
 *           dtab: T_oa_dyn, Q_solar[5], Q_x[5], T_oa_obs, lb_obs, ub_obs, time_of_day,
 *                 lb_prev, ub_prev
 *           state: 6 double rows (x[5], p_consumed)        action 6, obs popcount(mask)
 */
/*  HS_BEGIN  dpar: max_grid_power      dtab: grid cost of the event
 *            state: 5 double rows (pv_power, es_power, es_cost, pv_cost, grid_power = the
 *            reference's meta state, kept from step to step and across resets)
 *  HS_PV     dpar: obs_low, obs_high, 1/(high-low)    dtab: scaled profile value   action 1, obs 1
 *  HS_STORAGE dpar: lo, hi, eta_charge, eta_discharge, max_power, dt_hours, initial mean,
 *                 initial cost, max_storage_cost, 1/(hi-lo), 1/max_storage_cost,
 *                 1/eta_discharge, 1/dt_hours, 1/eta_charge     ipar: storage ordinal
 *            state: 2 double rows (SOC, current cost)                    action 1, obs 2
 *  HS_EV     dpar: the EV layout, then max_charge_cost, 60 / minutes_per_step, 1/max_charge_cost
 *            dtab: evaluation time, new time, hours_left[m], 1/hours_left[m]    itab: as EV
 *            state: n + 1 double rows (remaining kWh, current cost), words uint32 rows
 *                                                                        action 1, obs 7
 *  HS_DEVICES dpar: minutes_per_step / 60, obs_high[k], 1/obs_high[k]    ipar: k
 *            dtab: scaled row[k], unscaled row[k]                        action 1, obs k
 */
#define PGW_HS_MAX_COMPONENTS 8  /* components of one house, HS_BEGIN not counted */

typedef struct pgw_component {
  int32_t type;      /* pgw_component_type */
  int32_t agent;     /* owning agent (index into pgw_spec.agents) */
  int32_t flags;
  int32_t act_off;   /* first action row */
  int32_t obs_off;   /* first observation row */
  int32_t obs_dim;
  int32_t sd_off;    /* first row of the double state */
  int32_t si_off;    /* first row of the uint32 state */
  int32_t dtab_off;  /* offset (doubles) inside a row of the double event table */
  int32_t itab_off;  /* offset (int32) inside a row of the int event table */
  int32_t dpar_off;
  int32_t ipar_off;
} pgw_component;

/* One agent = ordered component list (gridworld/base.py:74-182 MultiComponentEnv) or a
 * single component (ComponentEnv, gridworld/base.py:12-71). */
typedef struct pgw_agent {
  int32_t comp_begin, comp_end; /* [begin, end) into pgw_spec.components */
  int32_t load_slot;            /* index of the feeder load the agent's P adds to, -1 = none
                                   (gridworld/multiagent_env.py:171-181, "bus" = load name)  */
  int32_t bus_node;             /* feeder node whose p.u. voltage is this agent's bus_voltage
                                   (opendss.py:173-186), -1 = not observed */
} pgw_agent;

/*
 * Compiled feeder: the network part of the OpenDSS circuit reduced to the load
 * branches (replaces the `Solve mode=snap` call of
 * gridworld/distribution_system/opendss.py:134 and the accessors at :156-186).
 * Complex arrays are interleaved (re, im) doubles, per unit on each branch's /
 * node's own voltage base and a 1 MVA power base.
 *   u      = u0 - Zbb * i(u)          fixed point over the nb load branches
 *   v_node = w  - Znb * i             all nn node voltages, magnitudes reported
 */
typedef struct pgw_feeder {
  int32_t nb;            /* load branches (IEEE-13: 14)                */
  int32_t nn;            /* electrical nodes (IEEE-13: 38)             */
  int32_t nl;            /* loads = addressable "bus" names (IEEE-13: 12) */
  int32_t max_iter;
  double tol;            /* max |du| (p.u.) convergence threshold      */
  const double* zbb;     /* [nb][nb] complex, row = output branch      */
  const double* u0;      /* [nb] complex                               */
  const double* znb;     /* [nn][nb] complex                           */
  const double* w;       /* [nn] complex                               */
  const int32_t* branch_load;  /* [nb] owning load                     */
  const double* branch_share;  /* [nb] 1/(branches of that load)       */
  const int32_t* branch_model; /* [nb] OpenDSS load model (1, 2, 5)    */
  const double* vminpu;        /* [nb]                                 */
  const double* vmaxpu;        /* [nb]                                 */
  /* grid-level reward hook (examples/marl/openai/train.py:51-88); unit_penalty 0 = off */
  int32_t penalty_node;
  double penalty_vlo, penalty_vhi, penalty_unit;
} pgw_feeder;

typedef struct pgw_spec {
  int32_t abi_version;   /* PGW_ABI_VERSION */
  int32_t num_envs;      /* E */
  int32_t num_agents;
  int32_t num_components;
  int32_t act_dim;       /* action rows per env  */
  int32_t obs_dim;       /* observation rows per env */
  int32_t sd_rows;       /* double state rows    */
  int32_t si_rows;       /* uint32 state rows    */
  int32_t num_storage;   /* rows of init_soc     */
  int32_t num_events;    /* rows of the event tables: event 0 = reset, event t+1 = step t */
  int32_t dtab_stride;   /* doubles per event row (even)  */
  int32_t itab_stride;   /* int32 per event row (multiple of 4) */
  int32_t dpar_len, ipar_len;
  const pgw_agent* agents;
  const pgw_component* components;
  const double* dpar;
  const int32_t* ipar;
  /* Event tables.  Row layout (doubles): [0] done flag of the event, [1] reserved,
   * [2 .. 2+nl) base kW per load, [2+nl .. 2+2nl) base kvar per load, then the
   * components' blocks at their dtab_off. */
  const double* dtab;    /* [num_events][dtab_stride] */
  const int32_t* itab;   /* [num_events][itab_stride] */
  const pgw_feeder* feeder; /* NULL = component-only env (no power flow) */
} pgw_spec;

typedef struct pgw_env pgw_env;

/* Fields readable with pgw_get (device destination, rows x E doubles unless noted). */
typedef enum pgw_field {
  PGW_FIELD_STATE_D = 0,   /* [sd_rows][E] double                                   */
  PGW_FIELD_STATE_I = 1,   /* [si_rows][E] uint32                                   */
  PGW_FIELD_AGENT_P = 2,   /* [A][E] kW, agent.real_power (base.py:51-55)           */
  PGW_FIELD_VOLTAGES = 3,  /* [nn][E] p.u. magnitudes (opendss.py:156-165)          */
  PGW_FIELD_VMIN = 4,      /* [E]                                                   */
  PGW_FIELD_VMAX = 5,      /* [E]                                                   */
  PGW_FIELD_VBUS = 6,      /* [A][E] voltage at each agent's bus node               */
  PGW_FIELD_PF_ITERS = 7,  /* [E] int32, negative = not converged within max_iter   */
  PGW_FIELD_EP_RETURN = 8, /* [A][E] reward summed since the last reset             */
  PGW_FIELD_PF_STATE = 9   /* [nbp][E] complex: last converged branch voltages (warm start;
                              nbp = branch count padded to 16 / a multiple of 32)   */
} pgw_field;

#define PGW_NUM_STATS 8
/* pgw_stats output: [0] env-steps since reset (E * steps), [1] sum of rewards of the
 * last step over envs and agents, [2] sum of episode returns, [3] sum of voltage
 * violations max(0, vlo - v, v - vhi) at the penalty node, [4] number of envs whose
 * last solve did not converge, [5] total power-flow iterations of the last solve,
 * [6] min voltage over envs and nodes, [7] max voltage. Additive entries 0..5 are
 * what the multi-GPU driver all-reduces (sum); 6/7 reduce with min/max. */

/* Create the device-side env batch.  Replaces MultiAgentEnv.__init__
 * (gridworld/multiagent_env.py:24-86) + OpenDSSSolver.__init__ (opendss.py:17-51)
 * once the host has compiled the scenario into tables.  All spec pointers are
 * HOST pointers; they are copied and need not outlive the call. */
int pgw_create(const pgw_spec* spec, pgw_env** out);
int pgw_destroy(pgw_env* env);

/* MultiAgentEnv.reset (multiagent_env.py:125-140): base-load power flow, agent
 * resets, first observation.  init_soc: device [num_storage][E] initial storage
 * (the reference draws it on the host RNG, energy_storage_env.py:82-84; parity
 * runs feed the same numbers) or NULL to keep each storage's configured mean.
 * obs: device [obs_dim][E]. */
int pgw_reset(pgw_env* env, const double* init_soc, double* obs, void* cuda_stream);

/* MultiAgentEnv.step (multiagent_env.py:151-212) for all E envs.
 * actions [act_dim][E] -> obs [obs_dim][E], rew [A][E], done [E] (uint8). */
int pgw_step(pgw_env* env, const double* actions, double* obs, double* rew,
             uint8_t* done, void* cuda_stream);

/* Same two calls with HOST buffers: results are on the host when the call returns (the stream is
 * synchronised) -- the end-to-end path.  Page-locked buffers are read and written in place by the
 * kernels (PGW_OPT_HOST_ZERO_COPY); pageable ones are staged with copies. */
int pgw_reset_host(pgw_env* env, const double* init_soc, double* obs, void* cuda_stream);
int pgw_step_host(pgw_env* env, const double* actions, double* obs, double* rew,
                  uint8_t* done, void* cuda_stream);

/* Float32 I/O: the same four calls with float actions [act_dim][E] and float observations
 * [obs_dim][E].  The arithmetic is unchanged (float64): actions are widened where they are read,
 * observations rounded to nearest where they are stored; init_soc, rewards and done flags keep
 * their types.  A handle may be driven in both forms; pgw_step keeps one captured graph per form. */
int pgw_reset_f32(pgw_env* env, const double* init_soc, float* obs, void* cuda_stream);
int pgw_step_f32(pgw_env* env, const float* actions, float* obs, double* rew, uint8_t* done,
                 void* cuda_stream);
int pgw_reset_host_f32(pgw_env* env, const double* init_soc, float* obs, void* cuda_stream);
int pgw_step_host_f32(pgw_env* env, const float* actions, float* obs, double* rew, uint8_t* done,
                      void* cuda_stream);

/* Stand-alone batched power flow on the handle's feeder: PowerFlowSolver.calculate_power_flow
 * (gridworld/distribution_system/powerflow.py:20-39) used without an env, as in
 * tests/distribution_system/test_opendss.py:7-16.  load_kw / load_kvar are device
 * [nl][E] TOTAL kW / kvar per load; results land in PGW_FIELD_VOLTAGES / VMIN / VMAX /
 * VBUS / PF_ITERS.  Does not touch the episode clock, rewards or component state. */
int pgw_pf_solve(pgw_env* env, const double* load_kw, const double* load_kvar, void* cuda_stream);

/* Copy an internal field to a device buffer of `bytes` bytes (must match exactly). */
int pgw_get(pgw_env* env, int field, void* dst, size_t bytes, void* cuda_stream);

/* Checkpoint / resume: overwrite an internal field from a device buffer (same sizes as
 * pgw_get; the voltage fields, agent power, episode returns and both state arrays are
 * writable) and set the episode clock (steps since reset, 0 <= steps < num_events).  The
 * reference has no env-level checkpointing (SURVEY.md section 5); restoring every field of
 * pgw_get plus the clock reproduces the trajectory bit for bit. */
int pgw_set(pgw_env* env, int field, const void* src, size_t bytes, void* cuda_stream);

/* The same for `row_count` consecutive rows of a [rows][num_envs] field (PGW_FIELD_STATE_D,
 * PGW_FIELD_STATE_I), starting at `row_begin`: src is a device buffer of row_count x num_envs
 * elements.  Per-env rosters of randomised charging stations (PGW_F_EV_PER_ENV) go in this way. */
int pgw_set_rows(pgw_env* env, int field, int row_begin, int row_count, const void* src, size_t bytes,
                 void* cuda_stream);
int pgw_set_clock(pgw_env* env, int steps, void* cuda_stream);

/* Replace the VALUES of the parameter block and of both event tables (host pointers; the
 * sizes and the component layout are those of pgw_create and cannot change; a NULL pointer
 * leaves that table alone).  Stream-ordered before the next pgw_reset / pgw_step; returns
 * after the host buffers have been consumed.  Replaces the roster re-sampling that
 * EVChargingEnv(randomize=True) does on every reset
 * (gridworld/agents/vehicles/ev_charging_env.py:154-157): the host draws the new roster,
 * rebuilds that station's parameter and event columns and calls this before pgw_reset. */
int pgw_update_tables(pgw_env* env, const double* dpar, int dpar_len, const double* dtab,
                      const int32_t* itab, void* cuda_stream);

/* Episode statistics (see PGW_NUM_STATS) reduced on the device into out[8] (device
 * pointer); the caller all-reduces it across ranks (one NCCL call per report). */
int pgw_stats(pgw_env* env, double* out, void* cuda_stream);

/* Steps taken since the last reset (host mirror of the device clock), -1 before reset. */
int pgw_clock(const pgw_env* env);
/* Number of kernels this handle has launched since creation (bench accounting). */
long long pgw_launch_count(const pgw_env* env);
/* CUDA graphs captured and instantiated since creation: pgw_step keeps ONE per handle and I/O form
 * (pgw_step / pgw_step_f32) however many different caller buffers it sees; pgw_step_host one per set
 * of host buffers and I/O form (at most 8). */
long long pgw_graph_captures(const pgw_env* env);
/* Resets taken so far.  The first reset of a handle initialises the state that the reference keeps
 * across episodes (Home-Steward meta state and storage cost, gridworld/base_hs.py:53-61); a
 * checkpoint carries the count so that a resumed handle does not repeat that (pgw_set_reset_count). */
long long pgw_reset_count(const pgw_env* env);
int pgw_set_reset_count(pgw_env* env, long long resets);
/* Runtime options (pgw_set_option): */
#define PGW_OPT_PF_KERNEL 0   /* 0 = FP64 SIMT fixed point (default); 1 = tcgen05 tensor-core
                                 fixed point (split-TF32 operands, FP32 accumulate in TMEM),
                                 feeders with <= 16 load branches; 2 = tcgen05 split-FP16 fixed
                                 point with the Z-bus resident in shared memory, feeders with
                                 <= 88 load branches (123-bus class)                          */
#define PGW_OPT_WARM_START 1  /* 1 (default): each solve starts from the env's previous solution */
#define PGW_OPT_GRAPHS 2      /* 1 (default): pgw_step replays ONE captured CUDA graph per handle, its kernel
                                 nodes re-pointed (cudaGraphExecKernelNodeSetParams) whenever the caller's
                                 (actions, obs, rew, done) pointers change; needs a non-default stream  */
#define PGW_OPT_PDL 3         /* 1 (default): the tcgen05 power-flow kernel of a step is launched as a
                                 programmatic dependent of the component kernel, which releases it
                                 early (griddepcontrol.launch_dependents): the power-flow prologue
                                 overlaps the component kernel */
#define PGW_OPT_CLIP_INIT_SOC 4  /* 1 (default): pgw_reset clips init_soc to each storage's range, what the
                                 reference does with an explicit init_storage (energy_storage_env.py:
                                 88-89); 0: used as given -- the reference does NOT clip the value it
                                 draws itself (:82-84), so a host that replays that draw turns it off */
#define PGW_OPT_PF_POLISH 5   /* full float64 sweeps of the fixed point run after the tcgen05 split-FP16
                                 solver (kernel 2) has converged -- followed by one more sweep over the
                                 rows the rewards and the agents read -- in the step solve of feeders with
                                 <= 16 load branches whose rewards read the fresh voltages (shared-penalty
                                 hook, examples/marl/openai/train.py:51-88).  Default 1: the penalty-node
                                 and agent-bus voltages then agree with the float64 solver to ~1e-9 p.u.,
                                 i.e. rewards within rtol 1e-5 / atol 2e-5.  0 = off (~5e-8 p.u.)       */
#define PGW_OPT_PF_TC_TOL_NANO 6 /* convergence threshold max|du| of the tcgen05 solvers in units of
                                 1e-9 p.u. (10 .. 100000).  Default: max(solver tol, 1e-7) -- float32 cannot
                                 resolve less --, and max(solver tol, 1e-6) where the float64 polish follows
                                 (PGW_OPT_PF_POLISH > 0): the polish contracts what the loop leaves behind */
#define PGW_OPT_FUSED 7       /* the whole step in one kernel (component steps -> tcgen05 power flow ->
                                 float64 polish -> rewards per 32-env tile), for feeders with <= 16 load
                                 branches, stock components and power-flow kernel 2: 0 = off, 1 (default)
                                 = when the batch is at most two tiles per SM (<= 9472 envs), 2 = always.
                                 Returns PGW_ERR_INVALID for 2 when the scenario is not eligible.        */
#define PGW_OPT_HOST_CHUNKS 8 /* env chunks the staged form of pgw_step_host pipelines (copy-in of chunk k+1 |
                                 kernels of chunk k | copy-out of chunk k-1 on streams of their own):
                                 0 (default) = automatic (4 once the observations of a step exceed 32 MB,
                                 else 1: a copy costs ~8 us of fixed latency), up to 8                    */
#define PGW_OPT_HOST_ZERO_COPY 9 /* 1 (default): when all four buffers of pgw_step_host are page-locked host
                                 memory the GPU can address (cudaHostAlloc / cudaHostRegister, torch
                                 pin_memory()), the step's kernels read and write them in place over PCIe;
                                 0, or pageable buffers: staged through device buffers with copies         */
int pgw_set_option(pgw_env* env, int option, int value);

/* Per-kernel device timing for benchmarks: when enabled, every launch of pgw_step is
 * bracketed by CUDA events on the launch stream.  pgw_get_timing synchronises the stream
 * and returns accumulated milliseconds since the last call / enable:
 * out[0] component kernel, out[1] power-flow kernel, out[2] number of steps timed. */
int pgw_set_timing(pgw_env* env, int enabled);
int pgw_get_timing(pgw_env* env, double* out3, void* cuda_stream);

const char* pgw_last_error(void);
int pgw_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PGW_H_ */
