// pool_plan.cpp - host-only view of the Newton schedule the library builds (tools/pool_gather_stats.py and
// tests/test_pool_chain.py compile it with g++ and read the plan through ctypes).
#include <algorithm>
#include <cstdio>
#include <cstring>

#include "../grid-fed-rl-gym_b200/csrc/gfr_image.hpp"

extern "C" {

// Builds the Newton image of `d` on `lanes` lanes.  info[0..3] = rows, positions, pool slots, length of the tail
// lists; then, when the caps allow, the 4 * positions record words go to `sched` and the tail lists to `tails`.
// Returns 0, or -1 when the library refuses the feeder (`err`, `err_cap` bytes, gets the complaint).
int pool_plan(const gfr_feeder_desc* d, int lanes, int* info, int32_t* sched, int sched_cap, int32_t* tails,
              int tails_cap, char* err, int err_cap) {
  gfr::FeederImage fi;
  const std::string complaint = gfr::build_feeder_image(d, lanes, GFR_SOLVER_NEWTON, &fi);
  if (!complaint.empty()) {
    if (err && err_cap > 0) std::snprintf(err, (size_t)err_cap, "%s", complaint.c_str());
    return -1;
  }
  const gfr::Layout& lay = fi.lay;
  const int32_t* ints = reinterpret_cast<const int32_t*>(fi.img.data());
  const int n_sched = 4 * lay.P;
  int n_tails = 0;
  for (int p = 0; p < lay.P; ++p) {
    const int32_t* r = ints + lay.o_sched + 4 * p;
    n_tails = std::max(n_tails, (r[1] & gfr::REC_LIST_MASK) + (int)((uint32_t)r[3] & 0xffffu));
  }
  info[0] = lay.nrows; info[1] = lay.P; info[2] = lay.n_pool; info[3] = n_tails;
  if (sched && sched_cap >= n_sched) std::memcpy(sched, ints + lay.o_sched, sizeof(int32_t) * n_sched);
  if (tails && tails_cap >= n_tails && n_tails > 0) std::memcpy(tails, ints + lay.o_child_slot, sizeof(int32_t) * n_tails);
  return 0;
}

}  // extern "C"
