// Internal launch-parameter blocks shared between api.cu and the kernel files.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pgw.h"

namespace pgw {

// The part of the static tables one agent's CTA needs (component descriptors and their
// parameter blocks), as 16-byte aligned ranges of the blob's comps / dpar / ipar sections.
struct AgentSlice {
  int c_lo, c_n;           // components [c_lo, c_lo + c_n)
  int d_lo, d_n;           // dpar doubles, d_lo and d_n even
  int i_lo, i_n;           // ipar int32, multiples of 4
  int pad0, pad1;
};

// One CTA of the component kernel: agent `agent`, env blocks j, j + n, j + 2n, ...  Heavy agents
// (buildings, EV stations) get more CTAs than light ones (PV, storage), so that the persistent
// CTAs of a launch finish together.  The agent's slice rides along: one 48-byte read per CTA.
struct CtaWork {
  int agent, j, n, pad;
  AgentSlice sl;
};

struct CompParams {
  int E, A;
  int e_lo, e_hi;          // env range of this launch (pgw_step_host pipelines chunks of envs); E stays
                           // the row stride of every per-env array
  unsigned int tickets;    // CTAs of all launches of the step's last kernel (clock advance)
  int event_mode;          // 0 = reset (event row 0), 1 = step (event row clock+1)
  int advance_clock;       // 1 when this kernel is the last one of the step (no feeder)
  int clip_init_soc;       // reset: clip init_soc to each storage's range (PGW_OPT_CLIP_INIT_SOC)
  int pdl_trigger;         // griddepcontrol.launch_dependents: 0 never, 1 after the clock read, 2 at the end
  int io32;                // 1: actions and obs are float arrays (the IO32 kernel instantiations), 0: double
  long long* phase_clk;    // PGW_PHASE_TIMERS builds only: [CTA][8] globaltimer at entry / exit + SM-clock stamps
  int owns_reward;         // 1 when no later kernel changes the reward (no feeder / no penalty)
  int has_house;           // 1: the scenario contains Home-Steward houses, 2: with telemetry
                           // (kernel variants)
  int ev_per_env;          // 1: a charging station runs on per-env rosters (kernel variant)
  int first_reset;         // reset only: first reset of the handle (state that the reference keeps
                           // across episodes gets its constructor value)
  // static tables, one contiguous 16-byte aligned blob: [agents | comps | dpar | ipar]
  const unsigned char* blob;
  int blob_bytes, off_comps, off_dpar, off_ipar;
  const CtaWork* work;        // [num_ctas] (device)
  int num_ctas;
  int max_cn, max_dn, max_in; // largest slice of any agent = the CTA's staging area
  const double* dtab;
  const int32_t* itab;
  int dstride, istride;
  const void* actions;      // [act_dim][E] double, or float under io32
  void* obs;               // [obs_dim][E] double, or float under io32
  double* rew;
  double* rew_copy;        // internal copy of the step's rewards (pgw_stats), written when this
                           // kernel owns the final reward (no feeder)
  uint8_t* done;
  double* sd;
  uint32_t* si;
  const double* init_soc;
  const double* vmin;
  const double* vmax;
  const double* vbus;
  double* agent_p;
  double* ep_ret;
  int* clock;
  unsigned int* ticket;
};

// Operand images + fp32 tables of the FP16 tensor-core power flow (powerflow_tc2.cu).
// blob: [B_hi | B_lo] (2 x part_bytes) | ncc x [Zn_hi | Zn_lo] at off_zn | tables at off_tab.
// Per-branch constants of the tc2 kernel, passed as a __grid_constant__ kernel parameter, laid
// out by PAIRS of branches (2q, 2q + 1) for the packed f32x2 arithmetic of the hot loop.
struct Tc2Consts {
  float4 pa[4 * 11];       // {Re u0 (2q), Re u0 (2q+1), Im u0 (2q), Im u0 (2q+1)}
  float4 pb[4 * 11];       // {vlo^2 (2q), vlo^2 (2q+1), vhi^2 (2q), vhi^2 (2q+1)}
  float4 pc[4 * 11];       // {g (2q), g (2q+1), h (2q), h (2q+1)}: (1, 0) = 1 / clamp(|u|^2),
                           // (0, 1) = 1 / |u| (constant-current load)
};

// Float64 tables of the polish sweeps (powerflow_tc2.cu, POLISH instantiations), passed as a
// __grid_constant__ kernel parameter: every entry is warp uniform, so the sweeps read them as
// constant-bank operands and shared memory only carries the per-env currents.
struct Tc2Polish {
  double2 zT[16 * 16];     // zT[j * 16 + k] = Zbb[k][j], zero padded
  float2 z32[16 * 16];     // the same / xscale in float32: the polish's float32 pre-sweep works on the
                           // scaled currents of the tensor-core loop
  double2 u0[16];
  double share[16];        // branch share x 1e-3 (kVA -> p.u. on 1 MVA), 0 for the padded branches
  double vlo2[16], vhi2[16];   // clamp band of |u|^2: model 1 [vmin^2, vmax^2], model 2 [1, 1]
  double dscale[16];       // node voltage = dscale x branch voltage (wye loads), else 0
  int model[16];
  unsigned rows;           // branches whose voltage the reward hook / the agents read (bit k)
  int pad;
};

struct Tc2Params {
  const unsigned char* blob;
  const Tc2Consts* consts; // host copy owned by the env handle
  const Tc2Polish* pconsts; // host copy owned by the env handle (polish only)
  int nch, ncc, nx, ntail, resident, part_bytes, off_zn, off_tab, tab_bytes, tmem_cols, any_m5;
  int t_share, t_bload, t_bagent, t_w, t_xnode, t_dnode, t_dscale, t_lptr, t_lidx,
      t_anode, t_vag, t_vtail;
  // FP64 polish of the converged branch voltages (feeders with <= 16 load branches, step solve
  // with the shared-penalty hook): `polish` full sweeps u <- u0 - Zbb i(u) in float64 on the
  // SIMT pipe after the tensor-core fixed point has converged, then one more sweep restricted to
  // the rows the reward hook and the agents read (Tc2Polish.rows), so that those voltages meet
  // the float64 tolerance (rewards 1e-5 relative / 2e-5 absolute).  0 = off.
  int polish, polish_ok, polish_row;   // polish_row: penalty node if it is NOT a wye-load node, else -1
  // Tables of the fused step kernel only (step_fused.cu), a section of their own behind the
  // shared ones: the Tc2Consts and Tc2Polish records byte for byte (the fused kernel reads them
  // from shared memory -- warp-uniform broadcasts -- instead of the parameter constant bank, whose
  // 7 kB are cold in every SM's constant cache at every launch) and, per agent, the load branch
  // whose wye node is the agent's bus (-1: none).  pen_slot: the same for the penalty node.
  // f_xz: Znb^T / xscale of the node-voltage expansion in float32, [16 branches][16 ncc slots]
  // (f_xz[k * 16 ncc + s] = Znb[xnode[s]][k] / xscale, zero padded).
  int off_ftab, ftab_bytes, f_kc, f_kp, f_aslot, f_xz, pen_slot;
  float xscale, descale1, descale2, tol;
};

struct PfParams {
  int E, A, nb, nn, nl, nbp, nnp, max_iter;
  int e_lo, e_hi;          // env range of this launch; E stays the row stride
  unsigned int tickets;    // CTAs of all launches of the step's last kernel (clock advance)
  double tol;
  int event_mode;          // 0 = reset (base load only, event row 0), 1 = step
  int advance_clock;
  int reward_hook;         // step with a shared voltage penalty: this kernel finishes the rewards
                           // (rew -= share, rew_copy, ep_ret); otherwise the component kernel did
  int warm_start;          // start from the previous solution kept in u_state
  int pdl;                 // launch as a programmatic dependent of the component kernel
  long long* phase_clk;    // PGW_PHASE_TIMERS builds only: [CTA][16] SM-clock stamps, else null
  // static tables, one contiguous 16-byte aligned blob (staged to shared memory by TMA
  // when it fits):  zbbT [nb][nbp] double2 (zbbT[j*nbp+k] = Zbb[k][j]) | u0 [nbp] double2 |
  // znbT [nb][nnp] double2 (znbT[k*nnp+n] = Znb[n][k]) | w [nnp] double2 |
  // share, vminpu, vmaxpu [nbp] double each | branch_load, branch_model [nbp] int32 each |
  // agent load_slot [A], agent bus_node [A] int32
  const unsigned char* blob;
  int blob_bytes, stage_blob;
  int off_u0, off_znbT, off_w, off_share, off_vmin, off_vmax, off_bload, off_bmodel, off_slot,
      off_node;
  double2* u_state;        // [nbp][E] last converged branch voltages (warm start)
  // tensor-core form (powerflow_tc.cu): operand images + fp32 tables, see TcLayout in api.cu
  const unsigned char* tc_blob;
  int tc_blob_bytes, tc_n2, tc_nnp8;
  int tc_off_b2, tc_off_u0, tc_off_w, tc_off_share, tc_off_vlo, tc_off_vhi, tc_off_bload,
      tc_off_bmodel, tc_off_slot, tc_off_node;
  float tc_tol;
  Tc2Params tc2;
  const double* agent_p;   // [A][E]
  const double* load_kw;   // [nl][E] stand-alone solve: total kW per load (else nullptr)
  const double* load_kvar; // [nl][E]
  const double* dtab;
  int dstride;
  double* vmag;            // [nn][E]
  double* vmin;
  double* vmax;
  double* vbus;            // [A][E]
  int32_t* iters;          // [E]
  double* rew;             // [A][E] (step only)
  double* rew_copy;        // [A][E] internal copy for pgw_stats
  double* ep_ret;          // [A][E]
  double* viol;            // [E] voltage violation at the penalty node
  int penalty_node;
  double pvlo, pvhi, punit;
  int* clock;
  unsigned int* ticket;
};

// One launch of the fused step kernel (step_fused.cu) over the envs [e_lo, e_hi).
struct FusedParams {
  CompParams c;            // component side: tables, event rows, caller buffers, state
  PfParams f;              // power-flow side: tc2 tables and images, voltages, penalty hook
  int C;                   // components per env
  int act_dim;             // action rows per env
  int sd_rows;             // double state rows per env
  int e_lo, e_hi;
  unsigned int tickets;    // CTAs of all launches of this step (the last one advances the clock)
  int stagger_cycles;      // CTA b delays the fetch of its first tile's actions by b x this many SM
                           // cycles (actions in host memory: requests served in tile order, so that
                           // the first tiles write their observations while the last ones still read)
  int pdl_trigger;         // 1: griddepcontrol.launch_dependents once the CTA has consumed the actions of
                           // its last tile (the next env chunk's launch may start: pgw_step_host)
  int event;               // >= 0: the step's event row, known to the host (direct launches, and graph
                           // replays whose node parameters are rewritten for new caller buffers anyway):
                           // the kernel skips the read of the device clock that the row's address would
                           // otherwise wait for.  -1: read the device clock (replays of a frozen graph).
};

struct StatsParams {
  int E, A, nn;
  const double* rew;
  const double* ep_ret;
  const double* viol;
  const int32_t* iters;
  const double* vmin;
  const double* vmax;
  const int* clock;
  double* out;             // [PGW_NUM_STATS]
};

cudaError_t launch_components(const CompParams& p, int smem_bytes, cudaStream_t s);
cudaError_t launch_powerflow(const PfParams& p, cudaStream_t s);
cudaError_t launch_powerflow_tc(const PfParams& p, cudaStream_t s);
cudaError_t launch_powerflow_tc2(const PfParams& p, cudaStream_t s);
size_t tc2_smem_bytes(const PfParams& p);
int tc2_grid(const PfParams& p);        // CTAs launch_powerflow_tc2 uses for p's env range
int fp64_grid(const PfParams& p);       // the same for launch_powerflow
int tc_grid(const PfParams& p);         // and for launch_powerflow_tc (whole batch only)
size_t tc2_polish_bytes(const PfParams& p);
bool tc2_polish_active(const PfParams& p);
int tc2_padded_chunks(int nch);      // instantiated tile width for nch chunks of 8 branches (0 = none)
constexpr int kTc2MaxChunks = 11;   // 88 load branches: B and A images fill shared memory
constexpr int kTcNb = 16;      // branch slots of the tensor-core kernel (IEEE-13 class feeders)
constexpr int kTcK3 = 96;      // 3 x 32: [x_hi | x_lo | x_hi] against [B_hi ; B_hi ; B_lo]
cudaError_t launch_stats(const StatsParams& p, cudaStream_t s);
cudaError_t launch_step_fused(const FusedParams& P, int grid, cudaStream_t s, bool programmatic = false);
size_t step_fused_smem_bytes(const FusedParams& P);
int step_fused_tiles(int envs);
bool is_step_fused_kernel(const void* func);   // graph node identification (api.cu)
bool is_component_kernel(const void* func);

}  // namespace pgw
