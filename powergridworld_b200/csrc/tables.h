// Static tables of one env batch, built on the host: pure functions of a pgw_spec that return the
// bytes the kernels read (layouts in internal.cuh) and the base launch parameters describing them,
// every pointer null.  No CUDA runtime calls: the caller uploads the tables and sets the pointers.
#pragma once
#include <string>
#include <vector>

#include "internal.cuh"

namespace pgw {

// "" when the spec is well formed (feeder tables aside), else the PGW_ERR_INVALID message
std::string validate_spec(const pgw_spec& s);

struct CompTables {
  std::vector<unsigned char> blob;   // [agents | comps | dpar | ipar], 16-byte aligned sections
  std::vector<CtaWork> work;         // every CTA of the heaviest agent, then the next agent, ...
  CompParams base{};
  bool need_scratch = false, need_scratch_reset = false;   // per-thread scratch of the building path
};
// cta_budget: CTAs to split over the agents (each gets 1 .. one per 64-env block)
CompTables build_comp_tables(const pgw_spec& s, int cta_budget);
// shared memory a component CTA stages: its agent's slice of the blob and one event row
int comp_staging_bytes(const CompParams& p);

struct FeederTables {
  std::string error;                 // "" or the PGW_ERR_INVALID message of a malformed feeder
  std::vector<unsigned char> blob;       // FP64 kernel (powerflow.cu)
  std::vector<unsigned char> tc_blob;    // split-TF32 kernel (powerflow_tc.cu), empty: feeder too large
  std::vector<unsigned char> tc2_blob;   // FP16 kernel (powerflow_tc2.cu) + the fused step's section
  PfParams base{};
  Tc2Consts tc2c{};
  Tc2Polish tc2p{};
};
// tc2_nch: tile width of the FP16 kernel for this feeder (tc2_padded_chunks), 0 = no tc2 tables
FeederTables build_feeder_tables(const pgw_spec& s, int tc2_nch);

// convergence threshold of the FP16 fixed point, from the float64 tolerance and the polish sweeps
float tc2_default_tol(double solver_tol, int polish);

}  // namespace pgw
