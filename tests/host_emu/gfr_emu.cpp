// gfr_emu.cpp - TEST INFRASTRUCTURE ONLY.  Compiles the device functions
// (grid-fed-rl-gym_b200/csrc/gfr_device.cuh) for the host so that control flow and arithmetic can be
// checked against the oracle in the build container, which has no GPU.  A group of LANES threads is
// emulated by LANES host threads that meet at a pthread barrier wherever the kernels synchronise the
// group, so the multi-lane schedules (register hand-off along a lane's path, pool slots between lanes)
// run as they do on the device.  Nothing in the package loads this; the product path is the CUDA
// library and nothing else.  Built by tests/host_emu/build.py into tests/host_emu/_build/ (git-ignored).
#include <pthread.h>

#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "../../grid-fed-rl-gym_b200/csrc/gfr_image.hpp"

using namespace gfr;

struct emu_env {
  DescCopy desc;
  FeederImage fi;
  EnvCfg cfg{};
  int solver = SOLVER_NEWTON;
  int lanes = 1;
  long long B = 0;
  std::vector<double> state, obs, bat_soc0;
};

namespace {

void team_barrier(void* ctx) { pthread_barrier_wait((pthread_barrier_t*)ctx); }

struct EmuSlot {
  std::vector<double> work;    // shared-memory slot
  std::vector<D2> mg;          // the global scratch of the slot
  std::vector<double> plocal;  // the per-thread injection array of a one-thread sweep on a small feeder
  explicit EmuSlot(const Layout& lay)
      : work(8 + (newton_slot_bytes(lay.n, lay.n_pool, 0) + sweep_slot_bytes(lay.n, 0, false, lay.n_tie)) / 8, 0.0),
        mg(newton_scratch_doubles(lay.P) / 2 + 1), plocal(SWEEP_P_LOCAL_MAX + 1, 0.0) {}
  template <class G> G group(const Layout& lay, int lane, EmuTeam* team) {
    G g;
    g.lane = lane; g.mask = 1u; g.red = nullptr; g.team = team;
    bind_slot(g, reinterpret_cast<unsigned char*>(work.data()), lay, mg.data(), plocal.data());
    return g;
  }
};

// run body(lane, team) on `lanes` host threads
void run_team(int lanes, const std::function<void(int, EmuTeam*)>& body) {
  pthread_barrier_t bar;
  pthread_barrier_init(&bar, nullptr, (unsigned)lanes);
  std::vector<double> red((size_t)lanes + 1, 0.0);
  EmuTeam team{lanes, team_barrier, &bar, red.data()};
  if (lanes == 1) { body(0, &team); pthread_barrier_destroy(&bar); return; }
  std::vector<std::thread> th;
  for (int l = 0; l < lanes; ++l) th.emplace_back([&, l] { body(l, &team); });
  for (auto& t : th) t.join();
  pthread_barrier_destroy(&bar);
}

template <int LANES>
void step_all(emu_env* e, const double* actions, const double* noise, const StepOut& o) {
  const Layout& lay = e->fi.lay;
  const int* simg = (const int*)e->fi.img.data();
  const double* dimg = (const double*)e->fi.img.data();
  EmuSlot slot(lay);
  run_team(LANES, [&](int lane, EmuTeam* team) {
    for (long long i = 0; i < e->B; ++i) {
      if (e->solver == SOLVER_NEWTON)
        step_instance<LANES, SOLVER_NEWTON>(slot.group<NGrp<LANES>>(lay, lane, team), lay, simg, dimg, e->cfg, i,
                                            e->state.data(), e->obs.data(), e->obs.data(), 0, actions, noise, o);
      else if (lay.n_tie)
        step_instance<LANES, SOLVER_SWEEP_TIES>(slot.group<SGrp<LANES>>(lay, lane, team), lay, simg, dimg, e->cfg, i,
                                                e->state.data(), e->obs.data(), e->obs.data(), 0, actions, noise, o);
      else
        step_instance<LANES, SOLVER_SWEEP>(slot.group<SGrp<LANES>>(lay, lane, team), lay, simg, dimg, e->cfg, i,
                                           e->state.data(), e->obs.data(), e->obs.data(), 0, actions, noise, o);
    }
  });
}

template <int LANES>
void solve_all(const FeederImage& fi, int solver, const EnvCfg& k, long long B, const double* p_inj, const SolOut& o) {
  const Layout& lay = fi.lay;
  const int* simg = (const int*)fi.img.data();
  const double* dimg = (const double*)fi.img.data();
  EmuSlot slot(lay);
  run_team(LANES, [&](int lane, EmuTeam* team) {
    for (long long i = 0; i < B; ++i) {
      if (solver == SOLVER_NEWTON)
        solve_instance<LANES, SOLVER_NEWTON>(slot.group<NGrp<LANES>>(lay, lane, team), lay, simg, dimg, k, i, p_inj, o);
      else if (lay.n_tie)
        solve_instance<LANES, SOLVER_SWEEP_TIES>(slot.group<SGrp<LANES>>(lay, lane, team), lay, simg, dimg, k, i, p_inj, o);
      else
        solve_instance<LANES, SOLVER_SWEEP>(slot.group<SGrp<LANES>>(lay, lane, team), lay, simg, dimg, k, i, p_inj, o);
    }
  });
}

bool lanes_ok(int lanes) { return lanes == 1 || lanes == 2 || lanes == 4 || lanes == 8 || lanes == 16; }

}  // namespace

extern "C" {

emu_env* emu_create(const gfr_feeder_desc* d, long long B, const gfr_env_cfg* c) {
  auto* e = new emu_env();
  e->lanes = c->solver.lanes > 0 ? c->solver.lanes : 1;
  if (!lanes_ok(e->lanes)) { delete e; return nullptr; }
  std::string err = build_feeder_image(d, e->lanes, c->solver.solver, &e->fi);
  if (!err.empty()) { delete e; return nullptr; }
  const Layout& lay = e->fi.lay;
  e->B = B;
  e->solver = c->solver.solver == GFR_SOLVER_NEWTON ? SOLVER_NEWTON : SOLVER_SWEEP;
  e->cfg = env_cfg_of(c);
  e->state.assign((size_t)B * lay.R, 0.0);
  e->obs.assign((size_t)B * lay.D, 0.0);
  e->bat_soc0.assign(d->bat_soc0, d->bat_soc0 + lay.Bt);
  Lanes<1> g; g.lane = 0; g.mask = 1u;
  for (long long i = 0; i < B; ++i)
    reset_instance<1>(g, lay, (const int*)e->fi.img.data(), (const double*)e->fi.img.data(), e->cfg, i,
                      e->state.data(), e->obs.data(), 0, e->fi.load_pq.data(), e->bat_soc0.data(),
                      nullptr, nullptr, 0.0, true, (long long)c->env_id_offset);
  return e;
}

void emu_destroy(emu_env* e) { delete e; }
double* emu_obs(emu_env* e) { return e->obs.data(); }
int emu_obs_dim(emu_env* e) { return e->fi.lay.D; }
// schedule facts, for the tests: rows, positions, pool slots, branches handed over in registers
void emu_schedule_info(emu_env* e, int* out4) {
  out4[0] = e->fi.lay.nrows; out4[1] = e->fi.lay.P; out4[2] = e->fi.lay.n_pool; out4[3] = e->fi.n_reg_edges;
}

void emu_reset(emu_env* e, const uint64_t* seeds, const uint8_t* mask, const double* noise,
               double start_time) {
  const Layout& lay = e->fi.lay;
  Lanes<1> g; g.lane = 0; g.mask = 1u;
  for (long long i = 0; i < e->B; ++i) {
    if (mask && !mask[i]) continue;
    reset_instance<1>(g, lay, (const int*)e->fi.img.data(), (const double*)e->fi.img.data(), e->cfg, i,
                      e->state.data(), e->obs.data(), 0, e->fi.load_pq.data(), e->bat_soc0.data(), seeds,
                      noise, start_time, false, 0);
  }
}

void emu_step(emu_env* e, const double* actions, const double* noise, const gfr_step_out* out) {
  switch (e->lanes) {
    case 1: step_all<1>(e, actions, noise, *out); break;
    case 2: step_all<2>(e, actions, noise, *out); break;
    case 4: step_all<4>(e, actions, noise, *out); break;
    case 8: step_all<8>(e, actions, noise, *out); break;
    case 16: step_all<16>(e, actions, noise, *out); break;
  }
}

int emu_solve(const gfr_feeder_desc* d, long long B, const double* p_inj, const gfr_solver_cfg* c,
              const gfr_sol_out* out) {
  const int lanes = c->lanes > 0 ? c->lanes : 1;
  if (!lanes_ok(lanes)) return -2;
  FeederImage fi;
  std::string err = build_feeder_image(d, lanes, c->solver, &fi);
  if (!err.empty()) return -1;
  const int solver = c->solver == GFR_SOLVER_NEWTON ? SOLVER_NEWTON : SOLVER_SWEEP;
  const EnvCfg k = env_cfg_of(c);
  switch (lanes) {
    case 1: solve_all<1>(fi, solver, k, B, p_inj, *out); break;
    case 2: solve_all<2>(fi, solver, k, B, p_inj, *out); break;
    case 4: solve_all<4>(fi, solver, k, B, p_inj, *out); break;
    case 8: solve_all<8>(fi, solver, k, B, p_inj, *out); break;
    case 16: solve_all<16>(fi, solver, k, B, p_inj, *out); break;
  }
  return 0;
}

void emu_noise_fill(long long B, int n_slots, const uint64_t* seeds, const uint64_t* draws, double* out) {
  for (long long i = 0; i < B; ++i)
    for (int s = 0; s < n_slots; ++s) out[i * n_slots + s] = noise_slot(seeds[i], draws[i], s);
}

}  // extern "C"
