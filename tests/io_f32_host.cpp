// TEST INFRASTRUCTURE ONLY -- not part of the product, never linked into libpgw_b200.so.
//
// Host build (g++ -ffp-contract=off) of the component arithmetic of
// powergridworld_b200/csrc/component_math.cuh with float32 actions and observations
// (AgentIOT<float, float>, what the IO32 kernels instantiate).  Same entry points and argument
// record as tests/emu/emu.cpp, whose float64 build is the reference of tests/test_io_f32_cpu.py.
#include "../powergridworld_b200/csrc/component_math.cuh"

extern "C" {

struct EmuArgs {
  int E, A;
  const pgw_agent* agents;
  const pgw_component* comps;
  const double* dpar;
  const int32_t* ipar;
  const double* drow;
  const int32_t* irow;
  const float* actions;
  float* obs;
  double* rew;
  double* agent_p;
  double* sd;
  uint32_t* si;
  const double* init_soc;
  int clip_init_soc;
  const double* vmin;
  const double* vmax;
  const double* vbus;
};

using IoF32 = pgw::AgentIOT<float, float>;

static double g_scratch[pgw::kScratchDoubles];

static IoF32 make_io(const EmuArgs* a) {
  IoF32 io;
  io.scr.p = g_scratch;
  io.scr.stride = 1;
  io.E = a->E; io.actions = a->actions; io.aE = a->E; io.ae0 = 0; io.obs = a->obs; io.sd = a->sd; io.si = a->si;
  io.init_soc = a->init_soc; io.clip_init_soc = a->clip_init_soc; io.vmin = a->vmin; io.vmax = a->vmax; io.vbus = a->vbus;
  io.dpar = a->dpar; io.ipar = a->ipar; io.drow = a->drow; io.irow = a->irow;
  return io;
}

static int g_first_reset = 1;
void emu_set_first_reset(int v) { g_first_reset = v; }

void emu_reset(const EmuArgs* a) {
  IoF32 io = make_io(a);
  for (int ag = 0; ag < a->A; ++ag)
    for (int e = 0; e < a->E; ++e) {
      if (pgw::is_house(a->agents[ag], a->comps))
        pgw::house_reset<true>(a->agents[ag], a->comps, io, e, g_first_reset != 0);
      else
        pgw::agent_reset<true>(a->agents[ag], a->comps, io, e);
      a->agent_p[(size_t)ag * a->E + e] = 0.0;
    }
}

void emu_step(const EmuArgs* a) {
  IoF32 io = make_io(a);
  for (int ag = 0; ag < a->A; ++ag)
    for (int e = 0; e < a->E; ++e) {
      double p, r;
      if (pgw::is_house(a->agents[ag], a->comps))
        pgw::house_step<true>(a->agents[ag], a->comps, io, e, p, r);
      else
        pgw::agent_step<true>(a->agents[ag], a->comps, io, e, p, r);
      a->agent_p[(size_t)ag * a->E + e] = p;
      a->rew[(size_t)ag * a->E + e] = r;
    }
}

}  // extern "C"
