// C entry points over the host-side table construction (powergridworld_b200/csrc/tables.cpp) for
// tests/test_host_tables.py: the tables of a spec and their named offsets, without a device.
#include <cstring>
#include <string>

#include "../powergridworld_b200/csrc/tables.h"

static pgw::CompTables g_comp;
static pgw::FeederTables g_feed;
static std::string g_err;

extern "C" {

// 0: tables built; -1: the spec is invalid (ht_error)
int ht_build(const pgw_spec* s, int cta_budget, int tc2_nch) {
  g_err = pgw::validate_spec(*s);
  if (!g_err.empty()) return -1;
  g_comp = pgw::build_comp_tables(*s, cta_budget);
  g_feed = s->feeder ? pgw::build_feeder_tables(*s, tc2_nch) : pgw::FeederTables{};
  g_err = g_feed.error;
  return g_err.empty() ? 0 : -1;
}

const char* ht_error() { return g_err.c_str(); }

// bytes of a table (comp, work, pf, tc, tc2, tc2c, tc2p) and their address
long ht_table(const char* name, const void** data) {
  auto out = [data](const void* p, size_t n) { *data = p; return (long)n; };
  if (!strcmp(name, "comp")) return out(g_comp.blob.data(), g_comp.blob.size());
  if (!strcmp(name, "work")) return out(g_comp.work.data(), g_comp.work.size() * sizeof(pgw::CtaWork));
  if (!strcmp(name, "pf")) return out(g_feed.blob.data(), g_feed.blob.size());
  if (!strcmp(name, "tc")) return out(g_feed.tc_blob.data(), g_feed.tc_blob.size());
  if (!strcmp(name, "tc2")) return out(g_feed.tc2_blob.data(), g_feed.tc2_blob.size());
  if (!strcmp(name, "tc2c")) return out(&g_feed.tc2c, sizeof(g_feed.tc2c));
  if (!strcmp(name, "tc2p")) return out(&g_feed.tc2p, sizeof(g_feed.tc2p));
  return -1;
}

// a field of the base launch parameters (c.* component kernel, f.* power flow, t.* tc2), NaN if unknown
double ht_value(const char* name) {
  const pgw::CompParams& c = g_comp.base;
  const pgw::PfParams& f = g_feed.base;
  const pgw::Tc2Params& t = f.tc2;
#define V(field) if (!strcmp(name, #field)) return (double)(field);
  V(c.off_comps) V(c.off_dpar) V(c.off_ipar) V(c.blob_bytes) V(c.num_ctas) V(c.tickets)
  V(c.max_cn) V(c.max_dn) V(c.max_in) V(c.dstride) V(c.istride)
  V(f.nb) V(f.nn) V(f.nl) V(f.nbp) V(f.nnp) V(f.blob_bytes) V(f.stage_blob)
  V(f.off_u0) V(f.off_znbT) V(f.off_w) V(f.off_share) V(f.off_vmin) V(f.off_vmax)
  V(f.off_bload) V(f.off_bmodel) V(f.off_slot) V(f.off_node) V(f.penalty_node) V(f.punit)
  V(t.nch) V(t.ncc) V(t.nx) V(t.ntail) V(t.part_bytes) V(t.off_zn) V(t.off_tab) V(t.tab_bytes)
  V(t.t_share) V(t.t_bload) V(t.t_bagent) V(t.t_w) V(t.t_xnode) V(t.t_dnode) V(t.t_dscale)
  V(t.t_lptr) V(t.t_lidx) V(t.t_anode) V(t.t_vag) V(t.t_vtail) V(t.polish) V(t.polish_ok)
  V(t.polish_row) V(t.off_ftab) V(t.ftab_bytes) V(t.f_kc) V(t.f_kp) V(t.f_aslot) V(t.f_xz)
  V(t.pen_slot) V(t.xscale) V(t.descale1) V(t.descale2)
#undef V
  return __builtin_nan("");
}

}  // extern "C"
