// gfr_emu_pq.cpp - TEST INFRASTRUCTURE ONLY.  The host emulation (see gfr_emu.cpp) of the solve with specified
// reactive power: solve_instance<LANES, SOLVER, SPEC_Q = true> of grid-fed-rl-gym_b200/csrc/gfr_device.cuh, bound
// to its instance slot as solve_pq_kernel binds it ((P, Q) pairs in the Newton scratch, 48 B per bus in the sweep
// slot), a group of LANES lanes run as that many host threads meeting at a pthread barrier.  Built by
// tests/host_emu/emu_pq.py into tests/host_emu/_build/ (git-ignored); nothing in the package loads it.
#include <pthread.h>

#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "../../grid-fed-rl-gym_b200/csrc/gfr_image.hpp"

using namespace gfr;

namespace {

void team_barrier(void* ctx) { pthread_barrier_wait((pthread_barrier_t*)ctx); }

template <class G> struct LanesOf;
template <int L> struct LanesOf<NGrp<L>> { static constexpr int value = L; };
template <int L> struct LanesOf<SGrp<L>> { static constexpr int value = L; };

// the shared-memory slot and the global scratch of one instance slot, sized for the Q kernels
struct EmuSlot {
  std::vector<double> work;
  std::vector<D2> mg;
  explicit EmuSlot(const Layout& lay)
      : work(8 + (newton_slot_bytes(lay.n, lay.n_pool, 0) + sweep_slot_bytes(lay.n, 0, false, lay.n_tie, true)) / 8, 0.0),
        mg(newton_scratch_doubles(lay.P, true) / 2 + 1) {}
  template <class G> G group(const Layout& lay, int lane, EmuTeam* team) {
    G g;
    g.lane = lane; g.mask = 1u; g.red = nullptr; g.team = team;
    bind_slot<LanesOf<G>::value, true>(g, reinterpret_cast<unsigned char*>(work.data()), lay, mg.data());
    return g;
  }
};

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
void solve_all(const FeederImage& fi, int solver, const EnvCfg& k, long long B, const double* p_inj, const double* q_inj,
               const SolOut& o) {
  const Layout& lay = fi.lay;
  const int* simg = (const int*)fi.img.data();
  const double* dimg = (const double*)fi.img.data();
  EmuSlot slot(lay);
  run_team(LANES, [&](int lane, EmuTeam* team) {
    for (long long i = 0; i < B; ++i) {
      if (solver == SOLVER_NEWTON)
        solve_instance<LANES, SOLVER_NEWTON, true>(slot.group<NGrp<LANES>>(lay, lane, team), lay, simg, dimg, k, i,
                                                   p_inj, o, q_inj);
      else if (lay.n_tie)
        solve_instance<LANES, SOLVER_SWEEP_TIES, true>(slot.group<SGrp<LANES>>(lay, lane, team), lay, simg, dimg, k, i,
                                                       p_inj, o, q_inj);
      else
        solve_instance<LANES, SOLVER_SWEEP, true>(slot.group<SGrp<LANES>>(lay, lane, team), lay, simg, dimg, k, i,
                                                  p_inj, o, q_inj);
    }
  });
}

}  // namespace

extern "C" {

// p_inj, q_inj [B, n] pu in ref bus order; 0 on success
int emu_solve_pq(const gfr_feeder_desc* d, long long B, const double* p_inj, const double* q_inj,
                 const gfr_solver_cfg* c, const gfr_sol_out* out) {
  const int lanes = c->lanes > 0 ? c->lanes : 1;
  FeederImage fi;
  std::string err = build_feeder_image(d, lanes, c->solver, &fi);
  if (!err.empty()) return -1;
  const int solver = c->solver == GFR_SOLVER_NEWTON ? SOLVER_NEWTON : SOLVER_SWEEP;
  const EnvCfg k = env_cfg_of(c);
  switch (lanes) {
    case 1: solve_all<1>(fi, solver, k, B, p_inj, q_inj, *out); return 0;
    case 2: solve_all<2>(fi, solver, k, B, p_inj, q_inj, *out); return 0;
    case 4: solve_all<4>(fi, solver, k, B, p_inj, q_inj, *out); return 0;
    case 8: solve_all<8>(fi, solver, k, B, p_inj, q_inj, *out); return 0;
    case 16: solve_all<16>(fi, solver, k, B, p_inj, q_inj, *out); return 0;
  }
  return -2;
}

}  // extern "C"
