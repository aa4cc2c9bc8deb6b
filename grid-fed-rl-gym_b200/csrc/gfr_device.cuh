// gfr_device.cuh - per-instance math of the batched GridEnvironment.step path.
//
// One "group" of LANES threads owns one feeder instance at a time: 1..32 lanes inside one warp
// (group barrier = __syncwarp) or, for large feeders, the whole CTA (64, 128, 256 lanes, barrier =
// __syncthreads).  The instance's working set lives in shared memory; the compiled feeder (the
// "image") is staged next to it once per CTA with one bulk (TMA) copy, or read from global memory
// when the group is CTA-wide.  Buses are numbered in LEVEL order: the host's leaf -> root
// elimination schedule (topology.compile_feeder), k = 0 being the root of the elimination tree.
// The passes over the tree run ROW by row: lane l takes schedule position row * LANES + l (Newton:
// a lane follows a path of the tree and hands a child's terms to its parent in registers; sweep:
// the (row, lane) record names the bus), so a lane only needs a group barrier when it reads what
// another lane wrote.
//
// The functions are __host__ __device__ so that tests/host_emu can run them on a CPU - a group of
// 1 - 16 lanes as that many host threads meeting at a barrier wherever the kernels synchronise -
// without a GPU.  That harness is test infrastructure; the shipped library only launches the
// __global__ kernels.
//
// Reference (paths under /root/reference/grid_fed_rl/):
//   Newton-Raphson        environments/power_flow.py:89-211  (polar; flat start; check-then-update)
//   Jacobian              environments/power_flow.py:213-295 (+ deviation D2, see DESIGN.md)
//   update                environments/power_flow.py:297-327
//   line flows / losses   environments/power_flow.py:329-358, :199-200
//   env step              environments/grid_env.py:410-619 and the dynamics it calls
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/gfr_b200.h"

#if defined(__CUDACC__)
#define GFR_HD __host__ __device__ __forceinline__
#else
#define GFR_HD inline
#endif

namespace gfr {

enum { SOLVER_SWEEP = 0, SOLVER_NEWTON = 1, SOLVER_SWEEP_TIES = 2 };   // TIES: the sweep with the compensation step compiled in
enum { BUS_SLACK = 0, BUS_PV = 1, BUS_PQ = 2 };
enum { GEN_SOLAR = 0, GEN_WIND = 1 };
// An instance's working set in shared memory:
//   Newton:  ef[n] (e + jf, 16 B per bus) | pool[4][n_pool] (16-byte fields)
//            The elimination runs on a SCHEDULE: row after row (leaf -> root), lane l of the group taking
//            position row * LANES + l.  The host lets a lane follow a path of the tree, so most buses are
//            eliminated right after one of their children on the same lane: that child's Schur terms
//            (L D^-1 U, L D^-1 r) and its branch's share of the parent's calculated injection stay in
//            REGISTERS, and the parent's correction comes back down the same way.  Only the other
//            children go through a pool slot (planned by the host: held from the child's row up to the
//            row that reads it - the sibling that absorbs it into its chain, or the parent; field 0 of a
//            slot planned for the back-substitution carries the correction on the way down).  D^-1 U and D^-1 r, only needed
//            again in the back-substitution, and the specified injections live in a per-slot scratch
//            in global memory, by position, that stays L2 resident; the back-substitution loads them
//            two rows ahead into registers.
//   sweep:   40 B per bus in three arrays: e + jf | Jr + jJi (branch current) | P
// Before the solve the same space (Newton: ef + pool; sweep: the J fields) carries the load /
// generator / battery powers into the per-position injection sums.
enum { F_E = 0, F_F = 1, F_SCRATCH = 2 };
enum { S_JR = 2, S_P = 4 };                      // field tags of the sweep accessors
enum { SCRATCH_FIELDS_SWEEP = 2 };
// bus flag bits (word z of a schedule record / word w of the sweep's topology record)
enum { FL_PQ = 1, FL_FROM_IS_PARENT = 2, FL_FIXED_VM = 4, FL_THETA = 8,     // PQ: |V| unknown; THETA: angle unknown
       FL_SLACK_PATH = 16,                                                // on the path slack -> root (slack included, root not)
       FL_C_REG = 32,                                                     // Newton: the bus eliminated just before on this lane is a child (the "heir"): its Schur terms are in registers
       FL_P_REG = 64,                                                     // Newton: this bus is its parent's heir: nothing goes through the pool, either way
       FL_VALID = 128,                                                    // the schedule position holds a bus
       FL_POOL_SHIFT = 8, FL_POOL_MASK = 0xFFF,                           // bits 8..19: the bus's pool slot
       FL_XSLOT_SHIFT = 20,                                               // bits 20..31: the slot its parent's correction arrives in
       REC_LIST_MASK = 0xFFFFF, REC_KIDX_SHIFT = 20 };                    // word y: tail list begin | 1 + slot this bus puts ITS correction in << 20
// record (persistent per-instance state) slots, in doubles
enum { R_TIME = 0, R_FREQ, R_WIND, R_TEMP, R_CLOUD, R_TOTAL_LOSSES, R_EPISODE_REWARD, R_SEED,
       R_DRAWS, R_COUNTS, R_BAT };   // soc[Bt] then bpow[Bt] from R_BAT on

struct alignas(16) D2 { double x, y; };
struct alignas(16) I4 { int x, y, z, w; };   // per-bus topology: parent, child list begin, end, flags
GFR_HD int pool_slot_of(int w) { return (w >> FL_POOL_SHIFT) & FL_POOL_MASK; }
// A schedule record (one per position p = row * lanes + lane, 16 bytes):
//   x = bus k | parent's k << 16 (indices into ef)      y = first entry of the bus's tail list | 1 + slot for its correction << 20
//   z = flags | pool slot << 8 | correction slot << 20   w = chain tails it gathers | 1 + slot it absorbs << 16
// The children handed over through the pool are summed along sibling chains (the host's plan): a child may
// ABSORB the partial sum of one sibling eliminated in an earlier row (add that sibling's slot to its own
// hand-off), and the bus gathers only the chain tails nobody absorbed, listed in child_slot.
// On the way down a bus with children behind pool slots writes its correction ONCE, into a slot planned for
// the back-substitution alone; every such child reads it there (z: correction slot).  0 in a "1 + slot" = none.
GFR_HD int rec_bus(const I4& t) { return (int)((unsigned)t.x & 0xFFFFu); }
GFR_HD int rec_parent(const I4& t) { return (int)((unsigned)t.x >> 16); }
GFR_HD int rec_list(const I4& t) { return t.y & REC_LIST_MASK; }
GFR_HD int rec_kids_x_slot(const I4& t) { return (int)((unsigned)t.y >> REC_KIDX_SHIFT) - 1; }
GFR_HD int x_slot_of(int z) { return (int)((unsigned)z >> FL_XSLOT_SHIFT); }
GFR_HD int rec_tails(const I4& t) { return (int)((unsigned)t.w & 0xFFFFu); }
GFR_HD int rec_absorb(const I4& t) { return (int)((unsigned)t.w >> 16) - 1; }
// Groups of 8 lanes and more sum along sibling chains: there a warp holds at most four groups, and a hub's pool
// children gathered on one lane kept the others waiting.  Smaller groups keep the parent gathering every pool child
// (no absorb step compiled in, no chains planned): measured on a B200, the absorb step cost IEEE-13 on 2 lanes 2.2 %
// and IEEE-34 on 2 lanes 0.4 %, more than their few gather iterations saved.
enum { CHAIN_MIN_LANES = 8 };
template <int LANES> GFR_HD constexpr bool sibling_chains() { return LANES >= CHAIN_MIN_LANES; }

// Where everything is inside the feeder image (ints / doubles counted from the image base)
// plus the sizes; passed as a kernel parameter (constant bank).
struct Layout {
  int n, nl, L, G, Bt, A, D, m, n_src, R, img_bytes, n_noise, n_pool, k_slack;
  int nrows, P;                  // schedule: rows and positions (Newton: rows x lanes; sweep: P = n, position = bus)
  int n_tie;                     // loop-closing lines (sweep only): m = n - 1 + n_tie
  int o_tie_ends, o_tie_ptr, o_tie_inc, o_tie_y, o_tie_z, o_tie_rating, o_tie_zinv;
  // by position, every image
  int o_sched, o_rank, o_rankp, o_branch_of_line, o_inj_ptr, o_inj_idx, o_gen_type;
  int o_gb, o_rating, o_vm_set;
  // Newton
  int o_child_ent, o_child_slot, o_gbd, o_f0;
  int o_kids;                    // CTA-wide groups: the pool slots of a position's first 8 chain tails, 16 bits each (one I4)
  // sweep (compact per-bus arrays)
  int o_topo, o_child_idx, o_rx;
  int o_rowrec, sw_rows;         // several lanes: one record per (row, lane) = (bus | parent << 16, child list begin, end, flags)
  // components
  int o_load_base, o_gen_cap, o_gen_p0, o_gen_p1, o_gen_p2, o_bat_cap, o_bat_rating, o_bat_eff, o_profile;
  double s_base, inv_s_base, load_p_sum;
};

struct EnvCfg {
  double dt, v_min, v_max, f_min, f_max, penalty, load_noise, tol, accel;
  int episode_length, stochastic_loads, weather_variation, max_it;
};

struct SolveStat {
  double max_mismatch;
  int iterations;
  int converged;
};

// The Newton scratch in global memory (D^-1 U, D^-1 r, specified injections: written and read back within the
// launch, every Newton iteration) must stay in L2 while the observation - four to five times as many bytes,
// written once - streams past it.  The observation goes out evict-first (__stcs); the scratch carries an L2
// evict-last policy (a 64-bit descriptor made once per thread with createpolicy) on its stores and loads.
// Loads are plain (weak) loads without L1 allocation: __ldcg would be a STRONG.GPU load here, ordered against
// every earlier store of the thread (measured: 3 x slower kernel).
GFR_HD uint64_t scratch_policy() {
#if defined(__CUDA_ARCH__)
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
#else
  return 0;
#endif
}
GFR_HD D2 ld_scratch(const D2* p, uint64_t pol) {
#if defined(__CUDA_ARCH__)
  D2 r;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(r.x), "=d"(r.y) : "l"(p), "l"(pol) : "memory");
  return r;
#else
  (void)pol;
  return *p;
#endif
}
GFR_HD void st_scratch(D2* p, const D2 v, uint64_t pol) {
#if defined(__CUDA_ARCH__)
  asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" ::"l"(p), "d"(v.x), "d"(v.y), "l"(pol) : "memory");
#else
  (void)pol;
  *p = v;
#endif
}
GFR_HD double ld_scratch1(const double* p, uint64_t pol) {
#if defined(__CUDA_ARCH__)
  double r;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(pol) : "memory");
  return r;
#else
  (void)pol;
  return *p;
#endif
}
GFR_HD void st_scratch1(double* p, double v, uint64_t pol) {
#if defined(__CUDA_ARCH__)
  asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(p), "d"(v), "l"(pol) : "memory");
#else
  (void)pol;
  *p = v;
#endif
}

// ----------------------------------------------------------------------------- group ops

// numpy's maximum / minimum: a NaN in either argument is the result
GFR_HD double max_nan(double v, double w) { return (w > v || w != w) ? w : v; }
GFR_HD double min_nan(double v, double w) { return (w < v || w != w) ? w : v; }
struct OpMaxNan { GFR_HD double operator()(double v, double w) const { return max_nan(v, w); } };
struct OpMinNan { GFR_HD double operator()(double v, double w) const { return min_nan(v, w); } };
struct OpMax { GFR_HD double operator()(double v, double w) const { return fmax(v, w); } };
struct OpMin { GFR_HD double operator()(double v, double w) const { return fmin(v, w); } };
struct OpSum { GFR_HD double operator()(double v, double w) const { return v + w; } };

// The threads that cooperate on one instance.  LANES <= 32: part of one warp, group barrier =
// __syncwarp(mask), reductions by shuffles.  LANES > 32: the whole CTA owns the instance ("one
// CTA per instance" for large feeders), barrier = __syncthreads(), reductions go warp-first and
// then through `red` (shared memory, LANES / 32 doubles).
#if !defined(__CUDACC__)
// host emulation (tests/host_emu): the lanes of a group are host threads that meet at a barrier
struct EmuTeam { int lanes; void (*barrier)(void*); void* ctx; double* red; };
#endif

template <int LANES>
struct Lanes {
  int lane;        // lane inside the group
  unsigned mask;   // LANES <= 32: the group's lanes inside its warp
  double* red;     // LANES > 32: cross-warp reduction scratch
#if !defined(__CUDACC__)
  EmuTeam* team = nullptr;
#endif
  GFR_HD void sync() const {
#if defined(__CUDA_ARCH__)
#ifdef GFR_STRESS
    // race hunting build (tests only): every lane dawdles a pseudo-random while before AND after each group
    // barrier, so an access that relies on lanes happening to run in step - instead of on the barrier - shows
    // up as a result that differs from the plain build's
    { unsigned h_ = (unsigned)clock() * 2654435761u + (unsigned)threadIdx.x * 40503u; __nanosleep((h_ >> 20) & 1023u); }
#endif
    if (LANES > 32) __syncthreads();
    else if (LANES > 1) __syncwarp(mask);
#ifdef GFR_STRESS
    { unsigned h_ = (unsigned)clock() * 2246822519u + (unsigned)threadIdx.x * 7919u; __nanosleep((h_ >> 21) & 511u); }
#endif
#elif !defined(__CUDACC__)
    if (LANES > 1 && team) team->barrier(team->ctx);
#endif
  }
  template <class Op>
  GFR_HD double reduce(double v, Op op) const {   // every lane gets the result
#if defined(__CUDA_ARCH__)
    if (LANES <= 32) {
#pragma unroll
      for (int o = LANES / 2; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(mask, v, o));
    } else {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
      __syncthreads();                              // the previous reduction has been read by everyone
      if ((lane & 31) == 0) red[lane >> 5] = v;
      __syncthreads();
      v = red[0];
#pragma unroll
      for (int w = 1; w < LANES / 32; ++w) v = op(v, red[w]);
    }
#elif !defined(__CUDACC__)
    if (LANES > 1 && team) {
      team->red[lane] = v;
      team->barrier(team->ctx);
      double r = team->red[0];
      for (int w = 1; w < LANES; ++w) r = op(r, team->red[w]);
      team->barrier(team->ctx);
      v = r;
    }
#endif
    return v;
  }
  GFR_HD double bcast(double v, int src) const {    // lane `src`'s value, to every lane
#if defined(__CUDA_ARCH__)
    if (LANES > 32) {
      __syncthreads();
      if (lane == src) red[0] = v;
      __syncthreads();
      v = red[0];
    } else if (LANES > 1) {
      v = __shfl_sync(mask, v, src, LANES);
    }
#elif !defined(__CUDACC__)
    if (LANES > 1 && team) {
      if (lane == src) team->red[0] = v;
      team->barrier(team->ctx);
      v = team->red[0];
      team->barrier(team->ctx);
    }
#endif
    return v;
  }
  GFR_HD double gmax_nan(double v) const { return reduce(v, OpMaxNan()); }   // NaN-propagating (numpy semantics)
  GFR_HD double gmin_nan(double v) const { return reduce(v, OpMinNan()); }
  GFR_HD double gmax(double v) const { return reduce(v, OpMax()); }
  GFR_HD double gmin(double v) const { return reduce(v, OpMin()); }
  GFR_HD double gsum(double v) const { return reduce(v, OpSum()); }
  GFR_HD int gsum(int v) const { return (int)reduce((double)v, OpSum()); }      // small counts: exact
  GFR_HD int gor(int v) const { return reduce(v ? 1.0 : 0.0, OpMax()) != 0.0; }
};

// sweep working set, 40 B per bus in three arrays: e + jf | Jr + jJi (branch current, then W) | P
template <int LANES>
struct SGrp : Lanes<LANES> {
  D2* efp;        // [n]
  D2* jrp;        // [n]
  double* pp;     // [n] specified injections
  D2* jt;         // [n_tie] tie currents (from -> to) of a weakly meshed feeder, then [n_tie] their loop mismatches
  int n;
  GFR_HD double& at(int, int k) const { return pp[k]; }                                   // S_P
  GFR_HD D2& at2(int field, int k) const { return field == F_E ? efp[k] : jrp[k]; }       // F_E | S_JR
  GFR_HD D2& ef(int k) const { return efp[k]; }
  GFR_HD double pspec(int k) const { return pp[k]; }
  GFR_HD void set_pspec(int k, double v) const { pp[k] = v; }
  GFR_HD double& scr(int j) const { return reinterpret_cast<double*>(jrp)[j]; }           // sources: the J array, flat (2 n doubles)
};

// Newton working set (see the layout note above)
// a pool entry is four 16-byte fields: c0, c1 (L D^-1 U rows), cc (L D^-1 r), fl (branch share of P, Q),
// stored field-major (field f of slot s at poolp[f * n_pool + s])
enum { POOL_D2 = 4 };
template <int LANES>
struct NGrp : Lanes<LANES> {
  D2* efp;        // [n]      shared, followed directly by the pool
  D2* poolp;      // [POOL_D2][n_pool] shared
  int np;         // n_pool
  double* pp;     // [P]      specified injections by position (global scratch, right after mg)
  D2* mg;         // [3][P]   GLOBAL scratch of this instance slot: rows of D^-1 U (2) and D^-1 r (1), field-major, by position
  uint64_t pol;   // L2 evict-last policy of the scratch
  GFR_HD D2& ef(int k) const { return efp[k]; }
  GFR_HD double pspec(int p) const { return ld_scratch1(pp + p, pol); }
  GFR_HD void set_pspec(int p, double v) const { st_scratch1(pp + p, v, pol); }
  GFR_HD double& scr(int j) const { return reinterpret_cast<double*>(efp)[j]; }   // ef + pool, flat
};

template <int LANES, int SOLVER> struct GroupOf { typedef NGrp<LANES> type; };
template <int LANES> struct GroupOf<LANES, SOLVER_SWEEP> { typedef SGrp<LANES> type; };
template <int LANES> struct GroupOf<LANES, SOLVER_SWEEP_TIES> { typedef SGrp<LANES> type; };

// bytes of shared memory one instance slot needs (0 if the sources do not fit the scratch)
GFR_HD size_t newton_slot_bytes(int n, int n_pool, int n_src) {
  if (n_src > 2 * n + 2 * POOL_D2 * n_pool) return 0;
  return (size_t)n * 16 + (size_t)n_pool * (16 * POOL_D2);
}
// doubles of global scratch per instance slot (Newton): D^-1 U, D^-1 r (48 B per position) + specified injections
// (a whole number of 128-byte lines per slot: a slot's lines can be dropped from L2 without touching a neighbour's)
GFR_HD size_t newton_scratch_doubles(int P) { return (((size_t)P * 6 + (((size_t)P + 1) / 2) * 2) + 15) & ~(size_t)15; }
// One thread per instance on a small feeder: the specified injections move to a per-thread local array (L1,
// interleaved by thread), 32 B per bus stay in shared memory - 40 % more resident instances per SM
enum { SWEEP_P_LOCAL_MAX = 20 };
GFR_HD bool sweep_p_local(int lanes, int n) { return lanes == 1 && n <= SWEEP_P_LOCAL_MAX; }
GFR_HD size_t sweep_slot_bytes(int n, int n_src, bool p_local = false, int n_tie = 0) {
  if (n_src > SCRATCH_FIELDS_SWEEP * n) return 0;
  const size_t units = ((size_t)n * (p_local ? 32 : 40) + 15) / 16 + 2 * (size_t)n_tie;   // 16-byte units, made odd: neighbouring instances'
  return (units | 1) * 16;                                // slots then start 4 banks apart (conflict-free 128-bit accesses)
}
// Points a group at its instance slot: `slot` in shared memory, `mg` its global scratch (Newton), `p_local` the
// thread's own array of SWEEP_P_LOCAL_MAX doubles (sweep, one lane; a caller that passes none points g.pp at its own)
template <int LANES>
GFR_HD void bind_slot(NGrp<LANES>& g, unsigned char* slot, const Layout& lay, D2* mg, double* = nullptr) {
  g.np = lay.n_pool;
  g.efp = reinterpret_cast<D2*>(slot);
  g.poolp = g.efp + lay.n;
  g.pp = reinterpret_cast<double*>(mg + 3 * (size_t)lay.P);
  g.mg = mg;
  g.pol = scratch_policy();
}
template <int LANES>
GFR_HD void bind_slot(SGrp<LANES>& g, unsigned char* slot, const Layout& lay, D2*, double* p_local = nullptr) {
  const int n = lay.n;
  g.efp = reinterpret_cast<D2*>(slot);
  g.jrp = g.efp + n;
  g.pp = reinterpret_cast<double*>(g.jrp + n);
  g.jt = g.jrp + n + (sweep_p_local(LANES, n) ? 0 : (n + 1) / 2);      // after the injections, when they live here
  g.n = n;
  // one thread per instance on a small feeder: the specified injections live in the thread's local array (the host
  // sized the shared-memory slot without them)
  if (sweep_p_local(LANES, n)) g.pp = p_local;
}


// Observation stores are evict-first (st.global.cs): nobody on the chip reads them again this launch, and the
// stream must not push the solver's L2-resident scratch out.
// One instance's row of the observation [B, D]: fp64 (default) or fp32 (opt-in; the reference declares float32,
// grid_env.py:346), in this step's buffer; `prev` reads the previous observation (another buffer when the caller
// bound two alternating ones).  Pairs (2i, 2i + 1) go out as one 16-byte (8-byte) store when the row starts on an
// even element.
struct ObsRow {
  double* o64; float* o32;
  const double* p64; const float* p32;
  bool pair_ok;
  GFR_HD void put(int i, double v) const {
#if defined(__CUDA_ARCH__)
    if (o32) __stcs(o32 + i, (float)v); else __stcs(o64 + i, v);
#else
    if (o32) o32[i] = (float)v; else o64[i] = v;
#endif
  }
  GFR_HD void put2(int i, double a, double b) const {     // i even
#if defined(__CUDA_ARCH__)
    if (pair_ok) {
      if (o32) __stcs(reinterpret_cast<float2*>(o32 + i), make_float2((float)a, (float)b));
      else __stcs(reinterpret_cast<double2*>(o64 + i), make_double2(a, b));
      return;
    }
#endif
    put(i, a); put(i + 1, b);
  }
  GFR_HD double prev(int i) const { return p32 ? (double)p32[i] : p64[i]; }
  GFR_HD bool same_buffer() const { return o32 ? (const float*)o32 == p32 : (const double*)o64 == p64; }
};
GFR_HD ObsRow obs_row(void* obs, const void* obs_prev, int f32, long long env, int D) {
  ObsRow r;
  const long long off = env * (long long)D;
  r.o64 = f32 ? nullptr : reinterpret_cast<double*>(obs) + off;
  r.o32 = f32 ? reinterpret_cast<float*>(obs) + off : nullptr;
  r.p64 = f32 ? nullptr : reinterpret_cast<const double*>(obs_prev) + off;
  r.p32 = f32 ? reinterpret_cast<const float*>(obs_prev) + off : nullptr;
  r.pair_ok = (off & 1LL) == 0;
  return r;
}

// 1 / x for a normal, finite x: hardware seed + two Newton steps (~1 ulp), no slow-path call.
GFR_HD double rcp_fast(double x) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = fma(r, fma(-x, r, 1.0), r);
  r = fma(r, fma(-x, r, 1.0), r);
  return r;
#else
  return 1.0 / x;
#endif
}

// sin / cos of a Newton angle correction.  Corrections are small: a Taylor pair is exact to
// < 1 ulp of 1.0 for |x| <= 0.25 (next terms x^17/17! < 2e-25, x^18/18! < 1e-26).  Larger steps
// (a diverging solve) are halved first and doubled back; nothing here calls a library slow path.
GFR_HD void sincos_small(double x, double* s, double* c) {
  if (fabs(x) <= 0.0078125) {
    // every update after the first: |x| <= 2^-7, the next terms x^9 / 9! and x^8 / 8! are below 1e-24
    const double x2 = x * x;
    *s = fma(x * x2, fma(x2, fma(x2, -1.0 / 5040.0, 1.0 / 120.0), -1.0 / 6.0), x);
    *c = fma(x2, fma(x2, fma(x2, -1.0 / 720.0, 1.0 / 24.0), -0.5), 1.0);
    return;
  }
  int halvings = 0;
  if (fabs(x) > 0.25) {
    if (!(fabs(x) <= 64.0)) x -= 6.283185307179586 * rint(x * 0.15915494309189535);   // garbage in, bounded out
    while (fabs(x) > 0.25 && halvings < 6) { x *= 0.5; ++halvings; }
  }
  const double x2 = x * x;
  double ps = -1.0 / 1307674368000.0;                 // -1/15!
  ps = fma(ps, x2, 1.0 / 6227020800.0);               //  1/13!
  ps = fma(ps, x2, -1.0 / 39916800.0);                // -1/11!
  ps = fma(ps, x2, 1.0 / 362880.0);                   //  1/9!
  ps = fma(ps, x2, -1.0 / 5040.0);                    // -1/7!
  ps = fma(ps, x2, 1.0 / 120.0);                      //  1/5!
  ps = fma(ps, x2, -1.0 / 6.0);                       // -1/3!
  double sn = fma(x * x2, ps, x);
  double pc = 1.0 / 20922789888000.0;                 //  1/16!
  pc = fma(pc, x2, -1.0 / 87178291200.0);             // -1/14!
  pc = fma(pc, x2, 1.0 / 479001600.0);                //  1/12!
  pc = fma(pc, x2, -1.0 / 3628800.0);                 // -1/10!
  pc = fma(pc, x2, 1.0 / 40320.0);                    //  1/8!
  pc = fma(pc, x2, -1.0 / 720.0);                     // -1/6!
  pc = fma(pc, x2, 1.0 / 24.0);                       //  1/4!
  pc = fma(pc, x2, -0.5);
  double cs = fma(x2, pc, 1.0);
  for (; halvings > 0; --halvings) {                  // double-angle back up
    const double s2 = 2.0 * sn * cs, c2 = fma(-2.0 * sn, sn, 1.0);
    sn = s2; cs = c2;
  }
  *s = sn; *c = cs;
}

// atan2(f, e) of a bus voltage.  In any state a feeder can be operated in e > 0 and |f / e| is a few
// degrees: the odd series in t = f / e to t^21 is exact to < 1 ulp for |t| <= 0.16 (next term
// t^23 / 23 < 3e-20); anything else takes the library call.
GFR_HD double atan2_bus(double f, double e) {
  if (e > 0.25 && e < 4.0) {
    const double t = f * rcp_fast(e);
    if (fabs(t) <= 0.16) {
      const double z = t * t;
      double p = 1.0 / 21.0;
      p = fma(p, z, -1.0 / 19.0);
      p = fma(p, z, 1.0 / 17.0);
      p = fma(p, z, -1.0 / 15.0);
      p = fma(p, z, 1.0 / 13.0);
      p = fma(p, z, -1.0 / 11.0);
      p = fma(p, z, 1.0 / 9.0);
      p = fma(p, z, -1.0 / 7.0);
      p = fma(p, z, 1.0 / 5.0);
      p = fma(p, z, -1.0 / 3.0);
      return fma(t * z, p, t);
    }
  }
  return atan2(f, e);
}

// ----------------------------------------------------------------------------- Philox4x32-10

struct U4 { uint32_t x, y, z, w; };

GFR_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

GFR_HD U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = mulhi32(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    uint32_t hi1 = mulhi32(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    U4 t;
    t.x = hi1 ^ c.y ^ k0; t.y = lo1; t.z = hi0 ^ c.w ^ k1; t.w = lo0;
    c = t;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c;
}

GFR_HD double u53(uint32_t hi, uint32_t lo) {   // (0,1) on a 2^-53 grid, never 0 or 1
  uint64_t k = ((uint64_t)(hi >> 5) << 26) + (uint64_t)(lo >> 6);
  return ((double)k + 0.5) * (1.0 / 9007199254740992.0);
}

// block q of the noise row keyed (seed, draw): q = 0 -> uniform in *a; q >= 1 -> two normals
GFR_HD void noise_block(uint64_t seed, uint64_t draw, uint32_t q, double* a, double* b) {
  U4 c; c.x = (uint32_t)draw; c.y = (uint32_t)(draw >> 32); c.z = q; c.w = 0u;
  U4 w = philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  double u1 = u53(w.x, w.y), u2 = u53(w.z, w.w);
  if (q == 0u) { *a = u1; *b = u2; return; }
  double rad = sqrt(-2.0 * log(u1));
  double sn, cs;
#if defined(__CUDA_ARCH__)
  sincospi(2.0 * u2, &sn, &cs);          // exact range reduction, no slow path
#else
  sincos(6.283185307179586 * u2, &sn, &cs);
#endif
  *a = rad * cs; *b = rad * sn;
}

// normal for noise slot s >= 1 (slot 0 is the uniform)
GFR_HD double noise_slot(uint64_t seed, uint64_t draw, int s) {
  double a, b;
  if (s == 0) { noise_block(seed, draw, 0u, &a, &b); return a; }
  int j = s - 1;
  noise_block(seed, draw, (uint32_t)(1 + j / 2), &a, &b);
  return (j & 1) ? b : a;
}

// ----------------------------------------------------------------------------- solvers

// Groups this wide read the feeder image from global memory (one CTA per instance).  Their row passes fetch what the
// NEXT row needs (its record, its branch / diagonal admittances, its packed pool-child record) while the present row
// computes - an L2 round trip per row otherwise (synthetic-1000: +8 %) - and they fetch index chains several
// positions at a time.  Measured and left off: the same row pipeline for warp-sized groups, whose image is in shared
// memory (IEEE-123 99.0 M -> 94.3 M, IEEE-34 306 M -> 284 M env-steps/s - the registers and moves cost more than the
// shared-memory latency they hide), and fetching the branch's two voltages one row ahead as well (synthetic-1000
// 5.91 M -> 5.64 M).
#ifndef GFR_WIDE_GROUP_MIN_LANES
#define GFR_WIDE_GROUP_MIN_LANES 64      // (the host emulation builds with 8 to walk these paths on its 8- and 16-lane teams)
#endif
template <int LANES> GFR_HD constexpr bool wide_group() { return LANES >= GFR_WIDE_GROUP_MIN_LANES; }

// Flat start (power_flow.py:103, :131): 1.0 at 0 rad, slack / PV buses at their set magnitude.
template <template <int> class G, int LANES>
GFR_HD void flat_start(const G<LANES>& g, const Layout& lay, const int* simg, const double* dimg) {
  const I4* sched = reinterpret_cast<const I4*>(simg + lay.o_sched);
  if (wide_group<LANES>()) {
    // image in global memory: four positions' records (and set points) per L2 round trip
    for (int p0 = g.lane; p0 < lay.P; p0 += 4 * LANES) {
      I4 t[4]; double vs[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int p = p0 + u * LANES;
        t[u].x = t[u].y = t[u].z = t[u].w = 0; vs[u] = 1.0;
        if (p < lay.P) { t[u] = sched[p]; vs[u] = dimg[lay.o_vm_set + p]; }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (!(t[u].z & FL_VALID)) continue;
        D2 v;
        v.x = (t[u].z & FL_FIXED_VM) ? vs[u] : 1.0;
        v.y = 0.0;
        g.ef(rec_bus(t[u])) = v;
      }
    }
  } else
  // warp-sized groups read a set point only where a position has one (the wide loop's form with one position per
  // round, which reads every set point, is unrolled differently by the compiler: 3 - 10 % more or fewer instructions)
  for (int p = g.lane; p < lay.P; p += LANES) {
    const I4 t = sched[p];
    if (!(t.z & FL_VALID)) continue;
    D2 v;
    v.x = (t.z & FL_FIXED_VM) ? dimg[lay.o_vm_set + p] : 1.0;
    v.y = 0.0;
    g.ef(rec_bus(t)) = v;
  }
  g.sync();
}

// Polar Newton-Raphson on a radial feeder.  Same iterates as the reference's dense solve:
// the Jacobian of a tree has one 2x2 block per bus and two per branch, so eliminating buses
// leaf -> root has no fill-in.  Unknowns per bus are (d theta, d|V| / |V|): scaling the
// |V| column removes every division from the assembly and leaves the update unchanged.
//   off-diagonal block J[i,j] = [[ al, ga ], [ -ga, al ]],
//        al = |Vi||Vj| (G_ij sin th_ij - B_ij cos th_ij), ga = |Vi||Vj| (G_ij cos th_ij + B_ij sin th_ij)
//   diagonal block  J[i,i]   = [[ -Q_i - B_ii |Vi|^2, P_i + G_ii |Vi|^2 ], [ P_i - G_ii |Vi|^2, Q_i - B_ii |Vi|^2 ]]
// with G_ij + jB_ij = -(g + jb) of the branch and everything written on e + jf = |V| e^{j theta}:
//   |Vi||Vj| cos th_ij = ei ej + fi fj,  |Vi||Vj| sin th_ij = fi ej - ei fj   (no trigonometry).
// The entries of a branch's two off-diagonal blocks are also that branch's terms of the calculated
// injections: P_k = G_kk |Vk|^2 + ga_k + sum_c gl_c,  Q_k = -B_kk |Vk|^2 + al_k + sum_c ll_c
// (ga, al: block J[k,p] of the bus's own branch; gl, ll: block J[k,c] of a child's branch), so the
// elimination pass gets the mismatch for free once each child hands (gl, ll) up with its Schur terms.
// Elimination of bus k (all its children done): D_k = J[k,k] - sum_c C_c, r_k = mismatch_k - sum_c cc_c,
//   M_k = D_k^-1 J[k,p], v_k = D_k^-1 r_k, and its contribution to the parent p:
//   C_k = J[p,k] M_k, cc_k = J[p,k] v_k.   Back-substitution: x_k = v_k - M_k x_p.
struct BranchT { double ga, al, gl, ll; };
// vk: the bus below the branch, vp: its parent, y: series g + jb
GFR_HD BranchT branch_terms(const D2 vk, const D2 vp, const D2 y) {
  const double a = fma(vk.x, vp.x, vk.y * vp.y), s = fma(vk.y, vp.x, -vk.x * vp.y);
  BranchT t;
  t.ga = fma(-y.x, a, -y.y * s); t.al = fma(-y.x, s, y.y * a);     // J[k,p]
  t.gl = fma(-y.x, a, y.y * s);  t.ll = fma(y.x, s, y.y * a);      // J[p,k] (th_pk = -th_kp)
  return t;
}

// Calls f(slot) with the pool slot of each of a position's chain tails in turn.  CTA-wide groups read their image
// from global memory: there the first 8 slots come packed in a record (kq) that travels one row ahead with the
// position's own record, which takes the list's L2 round trip off every row's critical path.
GFR_HD unsigned shr16_pair(unsigned lo, unsigned hi) { return (lo >> 16) | (hi << 16); }
template <int LANES, class F>
GFR_HD void for_each_tail(const I4& t, const I4& kq, const int* child_slot, F&& f) {
  const int npk = rec_tails(t);
  if (wide_group<LANES>() && npk <= 8) {
    unsigned w0 = (unsigned)kq.x, w1 = (unsigned)kq.y, w2 = (unsigned)kq.z, w3 = (unsigned)kq.w;
#pragma unroll 1
    for (int j = 0; j < npk; ++j) {
      const int slot = (int)(w0 & 0xffffu);
      w0 = shr16_pair(w0, w1); w1 = shr16_pair(w1, w2); w2 = shr16_pair(w2, w3); w3 >>= 16;
      f(slot);
    }
  } else {
    const int q0 = rec_list(t);
#pragma unroll 1
    for (int q = q0; q < q0 + npk; ++q) f(child_slot[q]);
  }
}

// What a row pass reads of each of its positions (`load(p)`: record, admittances, factors ...).  CTA-wide groups take
// it from registers filled while the previous row computed; warp-sized groups, whose image is in shared memory,
// load it when they need it.
template <int LANES, class T>
struct Ahead {
  T next = T();
  template <class Load> GFR_HD void first(const Load& load, int p) {
    if (wide_group<LANES>()) next = load(p);
  }
  // the data of position p; with more, the fetch of position p_next starts
  template <class Load> GFR_HD T take(const Load& load, int p, bool more, int p_next) {
    if (!wide_group<LANES>()) return load(p);
    const T now = next;
    if (more) next = load(p_next);
    return now;
  }
};
// a leaf -> root row pass (mismatch, elimination): the position's record, packed tail record (CTA-wide groups), and
// its branch's and diagonal admittances
struct RowIn { I4 t, kq; D2 y, yd; };

// A pool slot's hand-off to a parent, four fields: L D^-1 U (two rows), L D^-1 r, the branch's share of P, Q
GFR_HD void add_hand_off(const D2* e, int np, D2& h0, D2& h1, D2& hc, D2& hf) {
  const D2 c0 = e[0], c1 = e[np], cc = e[2 * np], fl = e[3 * np];
  h0.x += c0.x; h0.y += c0.y; h1.x += c1.x; h1.y += c1.y; hc.x += cc.x; hc.y += cc.y;
  hf.x += fl.x; hf.y += fl.y;
}
GFR_HD void put_hand_off(D2* e, int np, const D2 h0, const D2 h1, const D2 hc, const D2 hf) {
  e[0] = h0; e[np] = h1; e[2 * np] = hc; e[3 * np] = hf;
}

// max |mismatch| of the present voltages (power_flow.py:150-166), as a leaf -> root row pass on the elimination
// schedule: every branch is evaluated ONCE, by the bus below it, which keeps its own share (ga, al) and hands the
// parent's share (gl, ll) up - in registers to an heir's parent, through field 3 of its pool slot otherwise.
// Same arithmetic, term by term and in the same order, as the elimination pass.
template <int LANES>
GFR_HD double newton_mismatch(const NGrp<LANES>& g, const Layout& lay, const int* simg, const double* dimg) {
  const int nrows = lay.nrows, np = lay.n_pool;
  const I4* sched = reinterpret_cast<const I4*>(simg + lay.o_sched);
  const int* child_slot = simg + lay.o_child_slot;
  const D2* gb = reinterpret_cast<const D2*>(dimg + lay.o_gb);
  const D2* gbd = reinterpret_cast<const D2*>(dimg + lay.o_gbd);
  const I4* kids = reinterpret_cast<const I4*>(simg + (wide_group<LANES>() ? lay.o_kids : 0));
  double mm = 0.0;
  D2 hf; hf.x = hf.y = 0.0;                             // (gl, ll) of the bus this lane handled in the previous row
  double ps_next = g.pspec((nrows - 1) * LANES + g.lane);
  const auto row_in = [&](int p) {
    RowIn r = {sched[p], I4(), gb[p], gbd[p]};
    if (wide_group<LANES>()) r.kq = kids[p];
    return r;
  };
  Ahead<LANES, RowIn> ahead;
  ahead.first(row_in, (nrows - 1) * LANES + g.lane);
  for (int row = nrows - 1; row >= 0; --row) {
    const int p = row * LANES + g.lane;
    const RowIn in = ahead.take(row_in, p, row > 0, p - LANES);
    const I4 t = in.t;                                  // idle positions: record 0 -> bus 0, harmless
    const D2 vk = g.ef(rec_bus(t)), vp = g.ef(rec_parent(t));
    const double ps = ps_next;
    if (row > 0) ps_next = g.pspec(p - LANES);
    if (t.z & FL_VALID) {
      const double v2 = fma(vk.x, vk.x, vk.y * vk.y);
      const BranchT bt = branch_terms(vk, vp, in.y);
      if (!(t.z & FL_C_REG)) { hf.x = hf.y = 0.0; }
      for_each_tail<LANES>(t, in.kq, child_slot, [&](int slot) {
        const D2 fl = g.poolp[3 * np + slot];
        hf.x += fl.x; hf.y += fl.y;
      });
      const double P = fma(in.yd.x, v2, bt.ga) + hf.x, Q = fma(-in.yd.y, v2, bt.al) + hf.y;
      double aP = fabs(ps - P), aQ = fabs(Q);
      if ((t.z & (FL_PQ | FL_THETA)) != (FL_PQ | FL_THETA)) {   // slack: no equations; PV: no Q equation
        if (!(t.z & FL_THETA)) aP = 0.0;
        if (!(t.z & FL_PQ)) aQ = 0.0;
      }
      mm = max_nan(mm, max_nan(aP, aQ));
      hf.x = bt.gl; hf.y = bt.ll;
      if (sibling_chains<LANES>() && rec_absorb(t) >= 0) {                         // the partial of an earlier sibling's chain
        const D2 fl = g.poolp[3 * np + rec_absorb(t)];
        hf.x += fl.x; hf.y += fl.y;
      }
      if (!(t.z & FL_P_REG)) g.poolp[3 * np + pool_slot_of(t.z)] = hf;
    }
    g.sync();
  }
  return g.gmax_nan(mm);
}

// Back-substitution root -> leaf fused with the polar update (power_flow.py:297-327):
//   x_k = v_k - M_k x_parent (the root's M is 0: it has no branch), then
//   theta += a dtheta, |V| += a d|V|  <=>  V *= (1 + a x1) e^{j a x0}.
// x_parent is in the lane's registers when the bus is its parent's heir (the lane handled the parent one
// row earlier), else in field 0 of a pool slot (the parent put it there, once, for all such children).
// M and v come back from the global scratch (first iteration: M from the image), position by position -
// each lane reads back what it wrote itself.  Their L2 round trip is taken off the critical path by
// loading them TWO rows ahead into registers (the row loop is unrolled by two: even rows use the A set,
// odd rows the B set).
// D^-1 U (not in the first iteration: f0 holds it) and D^-1 r of a row into a register set.  Idle positions are
// loaded too (their scratch entries exist): no record is needed this early.
template <int LANES>
GFR_HD void load_mv(const NGrp<LANES>& g, int P, const D2* f0, int row, D2& m0, D2& m1, D2& v) {
  const int p = row * LANES + g.lane;
  if (!f0) { m0 = ld_scratch(g.mg + p, g.pol); m1 = ld_scratch(g.mg + P + p, g.pol); }
  v = ld_scratch(g.mg + 2 * P + p, g.pol);
}
struct BackIn { I4 t; D2 m0, m1; };                    // a position's record and, in the first iteration, D^-1 U
// One row: `in` is its position's record (and first-iteration D^-1 U), m0s / m1s / vs the register set loaded two
// rows earlier, refilled here for the row two ahead; hx is the correction of the bus this lane handled in the
// previous row.
template <int LANES>
GFR_HD void back_update_row(const NGrp<LANES>& g, int nrows, int P, const D2* f0, double accel, int row,
                            const BackIn& in, D2& hx, D2& m0s, D2& m1s, D2& vs) {
  const I4 t = in.t;
  const D2 e = g.efp[rec_bus(t)];
  D2 m0 = m0s, m1 = m1s, v = vs;
  if (f0) { m0 = in.m0; m1 = in.m1; }
  if (row + 2 < nrows) load_mv(g, P, f0, row + 2, m0s, m1s, vs);
  if (t.z & FL_VALID) {
    D2 x = hx;
    if (!(t.z & FL_P_REG)) x = g.poolp[x_slot_of(t.z)];
    v.x = fma(-m0.x, x.x, fma(-m0.y, x.y, v.x));
    v.y = fma(-m1.x, x.x, fma(-m1.y, x.y, v.y));
    if (rec_kids_x_slot(t) >= 0) g.poolp[rec_kids_x_slot(t)] = v;
    hx = v;
    double sn, cs;
    sincos_small(accel * v.x, &sn, &cs);
    const double sc = fma(accel, v.y, 1.0);
    D2 w;
    w.x = sc * fma(e.x, cs, -e.y * sn);
    w.y = sc * fma(e.x, sn, e.y * cs);
    g.efp[rec_bus(t)] = w;
  }
  g.sync();
}
template <int LANES>
GFR_HD void newton_back_update(const NGrp<LANES>& g, const Layout& lay, const int* simg, const D2* f0,
                               double accel) {
  const int nrows = lay.nrows, P = lay.P;
  const I4* sched = reinterpret_cast<const I4*>(simg + lay.o_sched);
  D2 a0, a1, av, b0, b1, bv;
  a0.x = a0.y = a1.x = a1.y = b0.x = b0.y = b1.x = b1.y = bv.x = bv.y = 0.0;
  D2 hx; hx.x = hx.y = 0.0;
  load_mv(g, P, f0, 0, a0, a1, av);
  if (nrows > 1) load_mv(g, P, f0, 1, b0, b1, bv);
  const auto back_in = [&](int p) {
    BackIn r = {sched[p], D2(), D2()};
    if (f0) { r.m0 = f0[2 * P + p]; r.m1 = f0[3 * P + p]; }
    return r;
  };
  Ahead<LANES, BackIn> ahead;
  ahead.first(back_in, g.lane);
  for (int row = 0; row < nrows; row += 2) {
    const int p = row * LANES + g.lane;
    back_update_row(g, nrows, P, f0, accel, row, ahead.take(back_in, p, row + 1 < nrows, p + LANES), hx, a0, a1, av);
    if (row + 1 < nrows)
      back_update_row(g, nrows, P, f0, accel, row + 1, ahead.take(back_in, p + LANES, row + 2 < nrows, p + 2 * LANES),
                      hx, b0, b1, bv);
  }
}

template <int LANES>
GFR_HD void newton_solve(const NGrp<LANES>& g, const Layout& lay, const int* simg,
                         const double* dimg, double tol, int max_it, double accel,
                         SolveStat* out) {
  const int nrows = lay.nrows, np = lay.n_pool, P = lay.P;
  const I4* sched = reinterpret_cast<const I4*>(simg + lay.o_sched);
  const int* child_slot = simg + lay.o_child_slot;   // pool slot of every child, indexed like child_ent
  const D2* gb = reinterpret_cast<const D2*>(dimg + lay.o_gb);      // branch series g, b by position (0 for the root)
  const D2* gbd = reinterpret_cast<const D2*>(dimg + lay.o_gbd);    // Re, Im of Y_kk by position
  const D2* f0 = lay.o_f0 >= 0 ? reinterpret_cast<const D2*>(dimg + lay.o_f0) : nullptr;   // flat-start factors
  const I4* kids = reinterpret_cast<const I4*>(simg + (wide_group<LANES>() ? lay.o_kids : 0));

  out->converged = 0;
  out->iterations = max_it;
  out->max_mismatch = INFINITY;
  double mm_prev = INFINITY, rate = 1.0;     // mismatch of the previous iterate, observed mm / mm_prev^2

  for (int it = 0; it < max_it; ++it) {
    double mm;
    if (it == 0 && f0 != nullptr) {
      // ---- first iteration: every instance starts from the same flat profile, so its calculated
      //      injections, its Jacobian and the whole elimination of it are properties of the feeder.
      //      The host factorised it once (image: D^-1, D^-1 U, J[p,k] and (P, Q) per position); only the
      //      right-hand side is instance data.
      mm = 0.0;
      for (int p = g.lane; p < P; p += LANES) {
        const int fl = sched[p].z;
        const D2 pc = f0[5 * P + p];
        double aP = fabs(g.pspec(p) - pc.x), aQ = fabs(pc.y);
        if (!(fl & FL_THETA)) aP = 0.0;
        if (!(fl & FL_PQ)) aQ = 0.0;
        const double loc = max_nan(aP, aQ);
        if (fl & FL_VALID) mm = max_nan(mm, loc);
      }
      mm = g.gmax_nan(mm);
      out->max_mismatch = mm;
      if (mm < tol) {                                   // checked before the update (:168-171)
        out->converged = 1;
        out->iterations = it + 1;
        break;
      }
      D2 hc; hc.x = hc.y = 0.0;                         // L v of the bus this lane eliminated in the previous row
      double ps_next = g.pspec((nrows - 1) * LANES + g.lane);     // the specified injection, one row ahead (an L2 round trip)
      struct F0In { I4 t, kq; D2 pc, i0, i1, lp; };   // record, packed tails, flat-profile (P, Q), D^-1 rows, (ll, gl)
      const auto f0_in = [&](int p) {
        F0In r = {sched[p], I4(), f0[5 * P + p], f0[p], f0[P + p], f0[4 * P + p]};
        if (wide_group<LANES>()) r.kq = kids[p];
        return r;
      };
      Ahead<LANES, F0In> ahead;
      ahead.first(f0_in, (nrows - 1) * LANES + g.lane);
      for (int row = nrows - 1; row >= 0; --row) {
        const int p = row * LANES + g.lane;
        const F0In in = ahead.take(f0_in, p, row > 0, p - LANES);
        const I4 t = in.t;
        const double ps = ps_next;
        if (row > 0) ps_next = g.pspec(p - LANES);
        if (t.z & FL_VALID) {
          if (!(t.z & FL_C_REG)) { hc.x = hc.y = 0.0; }
          for_each_tail<LANES>(t, in.kq, child_slot, [&](int slot) {
            const D2 cc = g.poolp[2 * np + slot];
            hc.x += cc.x; hc.y += cc.y;
          });
          const D2 sc = hc;
          double r0 = ps - in.pc.x - sc.x, r1 = 0.0 - in.pc.y - sc.y;
          if (!(t.z & FL_THETA)) r0 = 0.0;
          if (!(t.z & FL_PQ)) r1 = 0.0;
          D2 v;
          v.x = fma(in.i0.x, r0, in.i0.y * r1);
          v.y = fma(in.i1.x, r0, in.i1.y * r1);
          hc.x = fma(in.lp.x, v.x, in.lp.y * v.y);
          hc.y = fma(-in.lp.y, v.x, in.lp.x * v.y);
          if (sibling_chains<LANES>() && rec_absorb(t) >= 0) {
            const D2 cc = g.poolp[2 * np + rec_absorb(t)];
            hc.x += cc.x; hc.y += cc.y;
          }
          st_scratch(g.mg + 2 * P + p, v, g.pol);
          if (!(t.z & FL_P_REG)) g.poolp[2 * np + pool_slot_of(t.z)] = hc;
        }
        g.sync();
      }
      newton_back_update(g, lay, simg, f0, accel);
    } else {
      // ---- the iterate is expected to have converged (quadratic rate seen so far): a mismatch-only
      //      pass settles it without the elimination
      if (rate * mm_prev * mm_prev < 0.25 * tol) {
        mm = newton_mismatch(g, lay, simg, dimg);
        if (mm < tol) {
          out->max_mismatch = mm;
          out->converged = 1;
          out->iterations = it + 1;
          break;
        }
      }
      // ---- mismatch + assemble + eliminate, leaf -> root (power_flow.py:150-166, :213-295 with D2,
      //      then the solve of :187)
      mm = 0.0;
      int singular = 0;
      D2 h0, h1, hc, hf;                               // what the bus this lane eliminated in the previous row hands up
      h0.x = h0.y = h1.x = h1.y = hc.x = hc.y = hf.x = hf.y = 0.0;
      double ps_next = g.pspec((nrows - 1) * LANES + g.lane);     // the specified injection, one row ahead (an L2 round trip)
      const auto row_in = [&](int p) {
        RowIn r = {sched[p], I4(), gb[p], gbd[p]};
        if (wide_group<LANES>()) r.kq = kids[p];
        return r;
      };
      Ahead<LANES, RowIn> ahead;
      ahead.first(row_in, (nrows - 1) * LANES + g.lane);
      for (int row = nrows - 1; row >= 0; --row) {
        const int p = row * LANES + g.lane;
        const RowIn in = ahead.take(row_in, p, row > 0, p - LANES);
        const I4 t = in.t;
        const D2 vk = g.ef(rec_bus(t)), vp = g.ef(rec_parent(t)), yd = in.yd;
        const double ps = ps_next;
        if (row > 0) ps_next = g.pspec(p - LANES);
        if (t.z & FL_VALID) {
          const double v2 = fma(vk.x, vk.x, vk.y * vk.y);
          const BranchT bt = branch_terms(vk, vp, in.y);
          // children's contributions: plain sums, the heir first - it is what the lane still holds in h*
          if (!(t.z & FL_C_REG)) { h0.x = h0.y = h1.x = h1.y = hc.x = hc.y = hf.x = hf.y = 0.0; }
          for_each_tail<LANES>(t, in.kq, child_slot, [&](int slot) { add_hand_off(g.poolp + slot, np, h0, h1, hc, hf); });
          const D2 s0 = h0, s1 = h1, sc = hc, sf = hf;
          const double Pk = fma(yd.x, v2, bt.ga) + sf.x, Q = fma(-yd.y, v2, bt.al) + sf.y;
          D2 d0, d1, r;
          r.x = ps - Pk;
          r.y = 0.0 - Q;
          double aP = fabs(r.x), aQ = fabs(Q);
          r.x -= sc.x; r.y -= sc.y;
          d0.x = fma(-yd.y, v2, -Q) - s0.x;             // -Q - B v2
          d0.y = fma(yd.x, v2, Pk) - s0.y;              //  P + G v2
          d1.x = fma(-yd.x, v2, Pk) - s1.x;             //  P - G v2
          d1.y = fma(-yd.y, v2, Q) - s1.y;              //  Q - B v2
          double u00 = bt.al, u01 = bt.ga, u10 = -bt.ga, u11 = bt.al;
          if ((t.z & (FL_PQ | FL_THETA)) != (FL_PQ | FL_THETA)) {
            // a bus without the angle (slack) or magnitude (slack, PV) unknown: no equation, identity
            // row, no coupling
            if (!(t.z & FL_THETA)) { aP = 0.0; d0.x = 1.0; d0.y = 0.0; r.x = 0.0; u00 = 0.0; u01 = 0.0; }
            if (!(t.z & FL_PQ)) { aQ = 0.0; d1.x = 0.0; d1.y = 1.0; r.y = 0.0; u10 = 0.0; u11 = 0.0; }
          }
          mm = max_nan(mm, max_nan(aP, aQ));
          const double det = fma(d0.x, d1.y, -d0.y * d1.x);
          if (det == 0.0) singular = 1;                 // dgesv's exact-zero pivot (:188-190)
          const double inv = rcp_fast(det);
          const double i00 = d1.y * inv, i01 = -d0.y * inv, i10 = -d1.x * inv, i11 = d0.x * inv;
          D2 m0, m1, v;
          m0.x = fma(i00, u00, i01 * u10);
          m0.y = fma(i00, u01, i01 * u11);
          m1.x = fma(i10, u00, i11 * u10);
          m1.y = fma(i10, u01, i11 * u11);
          v.x = fma(i00, r.x, i01 * r.y);
          v.y = fma(i10, r.x, i11 * r.y);
          // handed to the parent: L M, L v, (gl, ll)
          h0.x = fma(bt.ll, m0.x, bt.gl * m1.x);
          h0.y = fma(bt.ll, m0.y, bt.gl * m1.y);
          h1.x = fma(-bt.gl, m0.x, bt.ll * m1.x);
          h1.y = fma(-bt.gl, m0.y, bt.ll * m1.y);
          hc.x = fma(bt.ll, v.x, bt.gl * v.y);
          hc.y = fma(-bt.gl, v.x, bt.ll * v.y);
          hf.x = bt.gl; hf.y = bt.ll;
          if (sibling_chains<LANES>() && rec_absorb(t) >= 0)                       // the partial of an earlier sibling's chain
            add_hand_off(g.poolp + rec_absorb(t), np, h0, h1, hc, hf);
          st_scratch(g.mg + p, m0, g.pol);               // needed again in the back-substitution only
          st_scratch(g.mg + P + p, m1, g.pol);
          st_scratch(g.mg + 2 * P + p, v, g.pol);
          if (!(t.z & FL_P_REG)) put_hand_off(g.poolp + pool_slot_of(t.z), np, h0, h1, hc, hf);
        }
        g.sync();
      }
      mm = g.gmax_nan(mm);
      out->max_mismatch = mm;
      if (mm < tol) {                                   // checked before the update (:168-171)
        out->converged = 1;
        out->iterations = it + 1;
        break;
      }
      if (g.gor(singular)) {
        out->iterations = it + 1;
        break;
      }
      newton_back_update(g, lay, simg, (const D2*)nullptr, accel);
    }
    {
      const double q = mm / (mm_prev * mm_prev);
      rate = (q > 1e-3 && q < 1e3) ? q : ((q >= 1e3) ? 1e3 : 1.0);
      mm_prev = mm;
    }
  }
#if defined(__CUDA_ARCH__)
  // The scratch of this solve is dead (the next instance of the slot rewrites it before reading): tell L2, so that
  // the dirty lines need not be written back to HBM when the observation stream pushes them out.  Every exit of the
  // loop above comes after a group-wide reduction, and every scratch read before that.  Measured on IEEE-123, 131 072
  // instances (0.59 GB of observation + state + outputs per launch; the evict-last hint alone changed nothing):
  // discarding the D^-1 U / D^-1 r lines writes 581 MB per launch at 98.1 M env-steps/s, discarding the injections'
  // lines too 565 MB at 97.8 M, keeping everything 1.02 GB at 99.2 M.
  {
    char* const base = reinterpret_cast<char*>(g.mg);
    const size_t bytes = ((size_t)P * 48) & ~(size_t)127;         // D^-1 U, D^-1 r only (whole lines), not the injections
    for (size_t off = (size_t)g.lane * 128; off < bytes; off += (size_t)LANES * 128)
      asm volatile("discard.global.L2 [%0], 128;" ::"l"(base + off) : "memory");
  }
#endif
}

// Backward / forward sweep (no counterpart in the reference, SURVEY F6; compared with the
// reference's Newton-Raphson at tight tolerance).  Constant-power injections P + j0, convergence on
// max(|de|, |df|) over buses.  The iteration is the classic one - branch currents from the present
// voltages, then voltages from the slack outwards - but it runs on the SAME center-rooted levels as
// the Newton elimination, which halves the sequential depth of a feeder whose slack sits at one end:
//   up   (leaf -> root)  A(k) = injected current of k (0 for the slack) + sum of A(children)
//   down (root -> leaf)  W(k) = W(parent) + z_k T(k),  T(k) = A(k) - [k on the slack -> root path] A(root)
//                        (what leaves subtree(k) through its branch; the slack's own injection is
//                        -A(root) by Kirchhoff), W = voltage relative to the root
//   fix  (every bus)     V(k) = V_slack - W(slack) + W(k)
//
// Weakly meshed feeders (lay.n_tie loop-closing lines, "ties"): the compensation method.  Every tie carries a
// current J (from -> to) that enters the sweep as a pair of bus injections (-J at the from-end, +J at the to-end);
// after the down pass the loop equations e = V_from - V_to - z_tie J are evaluated and J += Z_loop^-1 e, with the
// inverse loop-impedance matrix (constant: tree-path impedances shared by the loops + the ties' own) computed once
// by the host.  Convergence then needs max |dV| AND max |e| below the tolerance.
// TIES is a compile-time switch: the radial kernels do not carry the compensation code (4 more registers cost the
// IEEE-34 sweep its second CTA per SM: 270 M -> 238 M env-steps/s).
// adds to a the current the ties feed into bus k: + J at a to-end, - J at a from-end (nt = 0: nothing, no code)
GFR_HD void add_tie_current(const int* tie_ptr, const int* tie_inc, const D2* jt, int nt, int k, D2& a) {
  if (!nt) return;
  for (int q = tie_ptr[k]; q < tie_ptr[k + 1]; ++q) {
    const int e = tie_inc[q];
    const D2 j = jt[e >> 1];
    if (e & 1) { a.x += j.x; a.y += j.y; }
    else { a.x -= j.x; a.y -= j.y; }
  }
}
template <int LANES, bool TIES>
GFR_HD void sweep_solve(const SGrp<LANES>& g, const Layout& lay, const int* simg,
                        const double* dimg, double tol, int max_it, SolveStat* out) {
  const int n = lay.n, nrows = lay.sw_rows, ks = lay.k_slack, nt = TIES ? lay.n_tie : 0;
  const I4* topo = reinterpret_cast<const I4*>(simg + lay.o_topo);
  const I4* rowrec = reinterpret_cast<const I4*>(simg + (LANES > 1 ? lay.o_rowrec : 0));
  const int* child_idx = simg + lay.o_child_idx;
  const int* tie_ptr = simg + lay.o_tie_ptr;
  const int* tie_inc = simg + lay.o_tie_inc;
  const D2* rx = reinterpret_cast<const D2*>(dimg + lay.o_rx);
  const double vslack = dimg[lay.o_vm_set + ks];
  out->converged = 0;
  out->iterations = max_it;
  out->max_mismatch = INFINITY;
  if (nt) {
    D2 z0; z0.x = z0.y = 0.0;
    for (int i = g.lane; i < nt; i += LANES) g.jt[i] = z0;
    g.sync();
  }
  for (int it = 0; it < max_it; ++it) {
    if (LANES == 1) {
      // one thread per instance: buses are numbered parent before child, so a plain descending loop that
      // hands each subtree current to the parent needs no child lists (and no barriers)
      D2 z0; z0.x = z0.y = 0.0;
      for (int k = 0; k < n; ++k) g.at2(S_JR, k) = z0;
      double p_next = g.at(S_P, n - 1);                // the injections may live in local memory (L1 / L2): one bus ahead
      for (int k = n - 1; k >= 0; --k) {
        const I4 t = topo[k];
        const D2 v = g.at2(F_E, k);
        const double p_k = p_next;
        if (k > 0) p_next = g.at(S_P, k - 1);
        const double w = (t.w & FL_THETA) ? p_k * rcp_fast(fma(v.x, v.x, v.y * v.y)) : 0.0;
        D2 a = g.at2(S_JR, k);
        a.x = fma(w, v.x, a.x); a.y = fma(w, v.y, a.y);
        add_tie_current(tie_ptr, tie_inc, g.jt, nt, k, a);
        g.at2(S_JR, k) = a;
        if (k > 0) { D2& ap = g.at2(S_JR, t.x); ap.x += a.x; ap.y += a.y; }
      }
    } else {
      // several lanes: rows of at most LANES buses; a lane's record of the NEXT row (its bus, the parent, the child
      // list) is already in registers when the barrier falls - its position is known in advance
      I4 t_next = rowrec[(nrows - 1) * LANES + g.lane];
      for (int row = nrows - 1; row >= 0; --row) {
        const I4 t = t_next;
        if (row > 0) t_next = rowrec[(row - 1) * LANES + g.lane];
        if (t.w & FL_VALID) {
          const int k = t.x & 0xffff;
          const D2 v = g.at2(F_E, k);
          const double w = (t.w & FL_THETA) ? g.at(S_P, k) * rcp_fast(fma(v.x, v.x, v.y * v.y)) : 0.0;   // conj(S / V) = P V / |V|^2
          D2 a;
          a.x = w * v.x; a.y = w * v.y;
          add_tie_current(tie_ptr, tie_inc, g.jt, nt, k, a);
#pragma unroll 1
          for (int q = t.y; q < t.z; ++q) {
            const D2 ac = g.at2(S_JR, child_idx[q]);
            a.x += ac.x; a.y += ac.y;
          }
          g.at2(S_JR, k) = a;
        }
        g.sync();
      }
    }
    const D2 atot = g.at2(S_JR, 0);
    double mm = 0.0;
    // Several lanes: the root (level 0) is skipped - its W is 0 by definition, its voltage (the slack's set point when
    // the slack is the root, else rewritten by the fix-up pass) does not move, and its field keeps A(root) until the
    // next up pass, so no lane can find it overwritten before it has read it: two barriers less per iteration.
    if (LANES == 1) {
      for (int k = 0; k < n; ++k) {                    // one thread per instance: a single ascending loop over the buses
        const I4 t = topo[k];
        D2 w;
        w.x = 0.0; w.y = 0.0;
        if (k > 0) {
          D2 a = g.at2(S_JR, k);
          if (t.w & FL_SLACK_PATH) { a.x -= atot.x; a.y -= atot.y; }
          const D2 wp = g.at2(S_JR, t.x);
          const D2 z = rx[k];
          w.x = wp.x + fma(z.x, a.x, -z.y * a.y);
          w.y = wp.y + fma(z.x, a.y, z.y * a.x);
        }
        g.at2(S_JR, k) = w;
        if (ks == 0) {                                 // slack at the root: W is already V - V_slack
          const D2 vo = g.at2(F_E, k);
          D2 vn;
          vn.x = vslack + w.x; vn.y = w.y;
          const double de = fabs(vn.x - vo.x), df = fabs(vn.y - vo.y);
          const double loc = max_nan(de, df);
          mm = max_nan(mm, loc);
          g.at2(F_E, k) = vn;
        }
      }
    } else {
      I4 t_next = rowrec[(nrows > 1 ? 1 : 0) * LANES + g.lane];
      for (int row = 1; row < nrows; ++row) {
        const I4 t = t_next;
        if (row + 1 < nrows) t_next = rowrec[(row + 1) * LANES + g.lane];
        if (t.w & FL_VALID) {
          const int k = t.x & 0xffff, kp = (int)((unsigned)t.x >> 16);
          D2 a = g.at2(S_JR, k);
          if (t.w & FL_SLACK_PATH) { a.x -= atot.x; a.y -= atot.y; }
          D2 wp = g.at2(S_JR, kp);
          if (kp == 0) { wp.x = 0.0; wp.y = 0.0; }      // the root's field still holds A(root)
          const D2 z = rx[k];
          D2 w;
          w.x = wp.x + fma(z.x, a.x, -z.y * a.y);
          w.y = wp.y + fma(z.x, a.y, z.y * a.x);
          g.at2(S_JR, k) = w;
          if (ks == 0) {                               // slack at the root: W is already V - V_slack
            const D2 vo = g.at2(F_E, k);
            D2 vn;
            vn.x = vslack + w.x; vn.y = w.y;
            const double de = fabs(vn.x - vo.x), df = fabs(vn.y - vo.y);
            const double loc = max_nan(de, df);
            mm = max_nan(mm, loc);
            g.at2(F_E, k) = vn;
          }
        }
        g.sync();
      }
    }
    const D2 ws = g.at2(S_JR, ks);
    if (ks != 0)
    for (int k = g.lane; k < n; k += LANES) {
      D2 w = g.at2(S_JR, k);
      if (LANES > 1 && k == 0) { w.x = 0.0; w.y = 0.0; }
      const D2 vo = g.at2(F_E, k);
      D2 vn;
      vn.x = (vslack - ws.x) + w.x;
      vn.y = (0.0 - ws.y) + w.y;
      if (k == ks) { vn.x = vslack; vn.y = 0.0; }
      const double de = fabs(vn.x - vo.x), df = fabs(vn.y - vo.y);
      const double loc = max_nan(de, df);
      mm = max_nan(mm, loc);
      g.at2(F_E, k) = vn;
    }
    if (nt) {
      // loop equations of the ties with the new voltages, then the compensation step J += Z_loop^-1 e
      const int* ends = simg + lay.o_tie_ends;
      const D2* tz = reinterpret_cast<const D2*>(dimg + lay.o_tie_z);
      const D2* zinv = reinterpret_cast<const D2*>(dimg + lay.o_tie_zinv);
      D2* const et = g.jt + nt;
      g.sync();
      for (int i = g.lane; i < nt; i += LANES) {
        const D2 va = g.at2(F_E, ends[2 * i]), vb = g.at2(F_E, ends[2 * i + 1]), z = tz[i], j = g.jt[i];
        D2 e;
        e.x = (va.x - vb.x) - fma(z.x, j.x, -z.y * j.y);
        e.y = (va.y - vb.y) - fma(z.x, j.y, z.y * j.x);
        et[i] = e;
        const double de = fabs(e.x), df = fabs(e.y);
        const double loc = max_nan(de, df);
        mm = max_nan(mm, loc);
      }
      g.sync();
      for (int i = g.lane; i < nt; i += LANES) {
        D2 dj; dj.x = dj.y = 0.0;
        for (int q = 0; q < nt; ++q) {
          const D2 a = zinv[(size_t)i * nt + q], e = et[q];
          dj.x += fma(a.x, e.x, -a.y * e.y);
          dj.y += fma(a.x, e.y, a.y * e.x);
        }
        D2 j = g.jt[i];
        j.x += dj.x; j.y += dj.y;
        g.jt[i] = j;
      }
    }
    mm = g.gmax_nan(mm);
    g.sync();
    out->max_mismatch = mm;
    if (mm < tol) {
      out->converged = 1;
      out->iterations = it + 1;
      break;
    }
  }
}

// From -> to flow of the branch above the bus at position p (power_flow.py:329-358): P (pu), |S| (pu), series loss (pu)
// (the branch's record t and series admittance y already loaded)
template <class G>
GFR_HD void branch_flow_rec(const G& g, const I4 t, const D2 y, double* p_ft, double* s_abs, double* loss) {
  const D2 vk = g.ef(rec_bus(t)), vp = g.ef(rec_parent(t));
  const double de = vp.x - vk.x, df = vp.y - vk.y;                 // V_parent - V_k
  const double ir = y.x * de - y.y * df, ii = y.x * df + y.y * de;   // current parent -> k
  double P, Q;
  if (t.z & FL_FROM_IS_PARENT) {
    P = vp.x * ir + vp.y * ii; Q = vp.y * ir - vp.x * ii;    // V_p conj(I)
  } else {
    P = -(vk.x * ir + vk.y * ii); Q = -(vk.y * ir - vk.x * ii);    // V_k conj(-I)
  }
  *p_ft = P;
  *s_abs = sqrt(P * P + Q * Q);
  *loss = y.x * (de * de + df * df);                 // Re sum_i V_i conj((YV)_i), branch by branch
}

template <class G>
GFR_HD void branch_flow(const G& g, const Layout& lay, const int* simg, const double* dimg,
                        int p, double* p_ft, double* s_abs, double* loss) {
  branch_flow_rec(g, reinterpret_cast<const I4*>(simg + lay.o_sched)[p],
                  reinterpret_cast<const D2*>(dimg + lay.o_gb)[p], p_ft, s_abs, loss);
}

// From -> to flow of line `li` (ref order): a tree branch, or a tie of a weakly meshed feeder (I = y (V_from - V_to),
// S = V_from conj(I), power_flow.py:329-358).  Also gives the line's rating.
template <class G>
GFR_HD void line_flow(const G& g, const Layout& lay, const int* simg, const double* dimg,
                      int li, double* p_ft, double* s_abs, double* loss, double* rating) {
  const int pb = (simg + lay.o_branch_of_line)[li];
  if (pb >= 0) {
    branch_flow(g, lay, simg, dimg, pb, p_ft, s_abs, loss);
    *rating = dimg[lay.o_rating + pb];
    return;
  }
  const int i = -1 - pb;
  const int* ends = simg + lay.o_tie_ends;
  const D2 va = g.ef(ends[2 * i]), vb = g.ef(ends[2 * i + 1]);
  const D2 y = reinterpret_cast<const D2*>(dimg + lay.o_tie_y)[i];
  const double de = va.x - vb.x, df = va.y - vb.y;
  const double ir = y.x * de - y.y * df, ii = y.x * df + y.y * de;
  const double P = va.x * ir + va.y * ii, Q = va.y * ir - va.x * ii;
  *p_ft = P;
  *s_abs = sqrt(P * P + Q * Q);
  *loss = y.x * (de * de + df * df);
  *rating = dimg[lay.o_tie_rating + i];
}

// ----------------------------------------------------------------------------- solver entry (gfr_solve)

typedef gfr_sol_out SolOut;      // the caller's output table, as the C ABI declares it

template <int SOLVER, int LANES>
GFR_HD void run_solver(const NGrp<LANES>& g, const Layout& lay, const int* simg, const double* dimg,
                       const EnvCfg& cfg, SolveStat* st) {
  newton_solve(g, lay, simg, dimg, cfg.tol, cfg.max_it, cfg.accel, st);
}
template <int SOLVER, int LANES>
GFR_HD void run_solver(const SGrp<LANES>& g, const Layout& lay, const int* simg, const double* dimg,
                       const EnvCfg& cfg, SolveStat* st) {
  sweep_solve<LANES, SOLVER == SOLVER_SWEEP_TIES>(g, lay, simg, dimg, cfg.tol, cfg.max_it, st);
}

template <int LANES, int SOLVER>
GFR_HD void solve_instance(const typename GroupOf<LANES, SOLVER>::type& g, const Layout& lay,
                           const int* simg, const double* dimg, const EnvCfg& cfg, long long env,
                           const double* p_inj, const SolOut& o) {
  const int n = lay.n, m = lay.m;
  const int* rank = simg + lay.o_rank;
  const int* rankp = simg + lay.o_rankp;
  const double* pin = p_inj + env * n;
  for (int i = g.lane; i < n; i += LANES) g.set_pspec(rankp[i], pin[i]);
  g.sync();          // a position's injection is read by the lane that owns the position, not the one that owns ref bus i
  flat_start(g, lay, simg, dimg);
  SolveStat st;
  run_solver<SOLVER>(g, lay, simg, dimg, cfg, &st);
  for (int i = g.lane; i < n; i += LANES) {
    int k = rank[i];
    const D2 vv = g.ef(k);
    double e = vv.x, f = vv.y;
    if (o.bus_voltages) o.bus_voltages[env * n + i] = sqrt(e * e + f * f);
    if (o.bus_angles) o.bus_angles[env * n + i] = atan2_bus(f, e);
  }
  double loss = 0.0;
  for (int li = g.lane; li < m; li += LANES) {
    double P, S, ls, rating;
    line_flow(g, lay, simg, dimg, li, &P, &S, &ls, &rating);
    loss += ls;
    if (o.line_flows) o.line_flows[env * m + li] = P;
    if (o.line_loadings) o.line_loadings[env * m + li] = rating > 0.0 ? S * lay.s_base / rating : 0.0;
  }
  loss = g.gsum(loss);
  if (g.lane == 0) {
    if (o.losses) o.losses[env] = loss;
    if (o.max_mismatch) o.max_mismatch[env] = st.max_mismatch;
    if (o.converged) o.converged[env] = (uint8_t)st.converged;
    if (o.iterations) o.iterations[env] = st.iterations;
  }
  g.sync();
}

// ----------------------------------------------------------------------------- environment

typedef gfr_step_out StepOut;    // the caller's output table, as the C ABI declares it

GFR_HD bool finite_d(double x) { return fabs(x) <= 1.7976931348623157e308; }   // false for NaN / Inf

GFR_HD double clampd(double x, double lo, double hi) {    // np.maximum(lo, np.minimum(hi, x)), NaN stays NaN
  x = (x > hi) ? hi : x;
  return (x < lo) ? lo : x;
}

GFR_HD double hour_of(double t) { return fmod(t / 3600.0, 24.0); }   // (t / 3600) % 24, t >= 0

// SolarPVModel.get_power / WindTurbineModel.get_power (dynamics.py:120-142, :158-170)
GFR_HD double renewable_power(const Layout& lay, const int* simg, const double* dimg, int gi,
                              double hour, double wind, double temp, double cloud) {
  double cap = dimg[lay.o_gen_cap + gi];
  if (simg[lay.o_gen_type + gi] == GEN_SOLAR) {
    double area = dimg[lay.o_gen_p0 + gi], eff = dimg[lay.o_gen_p1 + gi];
    bool day = (hour >= 6.0) && (hour <= 18.0);
    double sun = day ? sin(3.141592653589793 * (hour - 6.0) / 12.0) : 0.0;
    double actual = (1000.0 * sun) * (1.0 - 0.8 * cloud);
    double dtc = temp - 25.0;
    double tf = 1.0 - 0.004 * (dtc > 0.0 ? dtc : 0.0);
    double p = actual * area * eff * tf;
    return p < cap ? p : cap;
  }
  double ci = dimg[lay.o_gen_p0 + gi], vr = dimg[lay.o_gen_p1 + gi], co = dimg[lay.o_gen_p2 + gi];
  if (wind < ci || wind > co) return 0.0;
  if (wind <= vr) {
    double q = (wind - ci) / (vr - ci);
    return cap * (q * q * q);
  }
  return cap;
}

// _update_weather (grid_env.py:653-681); u, z1..z3 are the four draws
GFR_HD void update_weather(double hour, double u, double z1, double z2, double z3, double* wind,
                           double* temp, double* cloud) {
  (void)u;   // irradiance is drawn but never read downstream (SURVEY A4)
  *wind = clampd(*wind + (0.0 + z1 * 0.5), 0.0, 30.0);
  *temp = (25.0 + 10.0 * sin(2.0 * 3.141592653589793 * (hour - 12.0) / 24.0)) + (0.0 + z2 * 2.0);
  *cloud = clampd(*cloud + (0.0 + z3 * 0.1), 0.0, 1.0);
}

template <int LANES, int SOLVER>
GFR_HD void step_instance(const typename GroupOf<LANES, SOLVER>::type& g, const Layout& lay,
                          const int* simg, const double* dimg, const EnvCfg& cfg, long long env,
                          double* state, void* obs, const void* obs_prev, int obs_f32, const double* actions,
                          const double* noise, const StepOut& o) {
  const int n = lay.n, m = lay.m, L = lay.L, G = lay.G, Bt = lay.Bt, A = lay.A, D = lay.D;
  double* rec = state + env * lay.R;
  const ObsRow ob = obs_row(obs, obs_prev, obs_f32, env, D);
  const double* act = actions + env * A;
  const int o_line = 2 * n, o_freq = 2 * n + 2 * m, o_gen = o_freq + 1 + 2 * L, o_bat = o_gen + G;

  // ---- action check (grid_env.py:424-428, 454-467): NaN / Inf -> -2 penalty, terminated,
  //      nothing advances.  A one-element action is replaced by 0.0 instead (SURVEY A1).
  int bad = 0;
  for (int a = g.lane; a < A; a += LANES) bad |= !finite_d(act[a]);
  bad = g.gor(bad);
  const bool zero_action = bad && (A == 1);
  if (zero_action) bad = 0;

  int step = ((const int32_t*)(rec + R_COUNTS))[0];
  int viol_count = ((const int32_t*)(rec + R_COUNTS))[1];
  double episode_reward = rec[R_EPISODE_REWARD];

  if (bad) {
    double vmax = -INFINITY, vmin = INFINITY;
    for (int i = g.lane; i < n; i += LANES) {
      double v = ob.prev(2 * i);
      vmax = fmax(vmax, v); vmin = fmin(vmin, v);
    }
    vmax = g.gmax(vmax); vmin = g.gmin(vmin);
    if (!ob.same_buffer())                               // alternating buffers: the unchanged state moves along
      for (int i = g.lane; i < D; i += LANES) ob.put(i, ob.prev(i));
    g.sync();
    {
      // get_observation() recomputes the renewable outputs from the clock and the weather
      // (grid_env.py:772-776); every other entry is state this path leaves alone
      const double hour = hour_of(rec[R_TIME]);
      for (int gi = g.lane; gi < G; gi += LANES)
        ob.put(o_gen + gi, renewable_power(lay, simg, dimg, gi, hour, rec[R_WIND], rec[R_TEMP], rec[R_CLOUD]));
    }
    if (g.lane == 0) {
      if (o.reward) o.reward[env] = -cfg.penalty * 2.0;
      if (o.terminated) o.terminated[env] = 1;
      if (o.truncated) o.truncated[env] = 0;
      if (o.error) o.error[env] = 1;
      if (o.converged) o.converged[env] = 0;
      if (o.iterations) o.iterations[env] = 0;
      if (o.max_voltage) o.max_voltage[env] = vmax;
      if (o.min_voltage) o.min_voltage[env] = vmin;
      if (o.losses) o.losses[env] = 0.0;
      if (o.max_mismatch) o.max_mismatch[env] = 0.0;
      if (o.violations) { for (int q = 0; q < 4; ++q) o.violations[env * 4 + q] = 0; }
      if (o.violation_count) o.violation_count[env] = viol_count;
      if (o.current_step) o.current_step[env] = step;
      if (o.episode_reward) o.episode_reward[env] = episode_reward;
    }
    if (o.noise_used)
      for (int s = g.lane; s < lay.n_noise; s += LANES) o.noise_used[env * lay.n_noise + s] = 0.0;
    return;
  }

  double t = rec[R_TIME], freq = rec[R_FREQ], wind = rec[R_WIND], temp = rec[R_TEMP],
         cloud = rec[R_CLOUD], total_losses = rec[R_TOTAL_LOSSES];
  const uint64_t seed = ((const uint64_t*)rec)[R_SEED];
  const uint64_t draw = ((const uint64_t*)rec)[R_DRAWS];
  const double dt = cfg.dt;
  const double* nz = noise ? noise + env * lay.n_noise : nullptr;

  // ---- batteries (grid_env.py:629-641; dynamics.py:189-220, 304-324)
  double soc_reward = 0.0;
  for (int b = g.lane; b < Bt; b += LANES) {
    double rating = dimg[lay.o_bat_rating + b], cap = dimg[lay.o_bat_cap + b],
           eff = dimg[lay.o_bat_eff + b];
    double soc = rec[R_BAT + b], cur = rec[R_BAT + Bt + b];
    double cmd = (zero_action ? 0.0 : act[b]) * rating;
    if (cmd > 0.0) {
      double lim = cmd < rating ? cmd : rating;
      double en = lim * dt / 3600.0, room = soc * cap * eff;
      en = en < room ? en : room;
      cur = en * 3600.0 / dt;
      soc = soc - en / (cap * eff);
    } else if (cmd < 0.0) {
      double lim = -cmd < rating ? -cmd : rating;
      double en = lim * dt / 3600.0, room = ((1.0 - soc) * cap) / eff;
      en = en < room ? en : room;
      cur = -(en * 3600.0 / dt);
      soc = soc + en * eff / cap;
    }
    rec[R_BAT + b] = soc; rec[R_BAT + Bt + b] = cur;
    ob.put(o_bat + 2 * b, soc); ob.put(o_bat + 2 * b + 1, cur);
    g.scr(L + G + b) = cur;
    soc_reward += (soc >= 0.2 && soc <= 0.8) ? 1.0 : -5.0;
  }
  // ---- clock, weather (grid_env.py:470-471, 653-681)
  t += dt;
  step += 1;
  const double hour = hour_of(t);
  double z_load0 = 0.0;
  if (cfg.weather_variation || (cfg.stochastic_loads && !nz)) {
    double u, z1, z2, z3, dummy;
    if (nz) { u = nz[0]; z1 = nz[1]; z2 = nz[2]; z3 = nz[3]; }
    else if (LANES >= 4) {
      // blocks 0..2 on lanes 0..2, shared by broadcast (one Philox + Box-Muller deep instead of three)
      double a = 0.0, b = 0.0;
      if (g.lane < 3) noise_block(seed, draw, (uint32_t)g.lane, &a, &b);
      u = g.bcast(a, 0); z1 = g.bcast(a, 1); z2 = g.bcast(b, 1); z3 = g.bcast(a, 2); z_load0 = g.bcast(b, 2);
      dummy = 0.0;
    } else {
      noise_block(seed, draw, 0u, &u, &dummy);
      noise_block(seed, draw, 1u, &z1, &z2);
      noise_block(seed, draw, 2u, &z3, &z_load0);
    }
    if (cfg.weather_variation) update_weather(hour, u, z1, z2, z3, &wind, &temp, &cloud);
    if (o.noise_used && g.lane == 0) {
      double* nu = o.noise_used + env * lay.n_noise;
      nu[0] = u; nu[1] = z1; nu[2] = z2; nu[3] = z3;
    }
  } else if (o.noise_used && g.lane == 0) {
    double* nu = o.noise_used + env * lay.n_noise;
    nu[0] = nu[1] = nu[2] = nu[3] = 0.0;
  }
  // ---- renewables (dynamics.py:120-170) and curtailment (grid_env.py:643-651)
  double tot_ren = 0.0, tot_used = 0.0;
  for (int gi = g.lane; gi < G; gi += LANES) {
    double p = renewable_power(lay, simg, dimg, gi, hour, wind, temp, cloud);
    double curtail = ((zero_action ? 0.0 : act[Bt + gi]) + 1.0) / 2.0;
    ob.put(o_gen + gi, p);
    g.scr(L + gi) = p * curtail;
    tot_ren += p;
    tot_used += p - p * (1.0 - curtail);
  }
  // ---- loads (dynamics.py:54-75)
  if (cfg.stochastic_loads) {
    int hi = (int)hour;
    int nx = (hi + 1) % 24;
    double frac = hour - (double)hi;
    double mult = dimg[lay.o_profile + hi] * (1.0 - frac) + dimg[lay.o_profile + nx] * frac;
    if (nz) {
      for (int l = g.lane; l < L; l += LANES) {
        double z = nz[4 + l];
        double pl = dimg[lay.o_load_base + l] * (mult * (1.0 + (0.0 + cfg.load_noise * z))) * 1.0;
        g.scr(l) = pl > 0.0 ? pl : 0.0;
        if (o.noise_used) o.noise_used[env * lay.n_noise + 4 + l] = z;
      }
    } else {
      // slot 4 + l is normal j = 3 + l: block 1 + j / 2, component j & 1
      if (g.lane == 0 && L > 0) {
        double pl = dimg[lay.o_load_base] * (mult * (1.0 + (0.0 + cfg.load_noise * z_load0))) * 1.0;
        g.scr(0) = pl > 0.0 ? pl : 0.0;
        if (o.noise_used) o.noise_used[env * lay.n_noise + 4] = z_load0;
      }
      for (int q = 3 + g.lane; 2 * q - 5 < L; q += LANES) {
        double za, zb;
        noise_block(seed, draw, (uint32_t)q, &za, &zb);
        int l = 2 * q - 5;
        double pl = dimg[lay.o_load_base + l] * (mult * (1.0 + (0.0 + cfg.load_noise * za))) * 1.0;
        g.scr(l) = pl > 0.0 ? pl : 0.0;
        if (o.noise_used) o.noise_used[env * lay.n_noise + 4 + l] = za;
        if (l + 1 < L) {
          pl = dimg[lay.o_load_base + l + 1] * (mult * (1.0 + (0.0 + cfg.load_noise * zb))) * 1.0;
          g.scr(l + 1) = pl > 0.0 ? pl : 0.0;
          if (o.noise_used) o.noise_used[env * lay.n_noise + 4 + l + 1] = zb;
        }
      }
    }
  } else {
    for (int l = g.lane; l < L; l += LANES) {
      g.scr(l) = dimg[lay.o_load_base + l];
      if (o.noise_used) o.noise_used[env * lay.n_noise + 4 + l] = 0.0;
    }
  }
  g.sync();
  // ---- injections per bus (grid_env.py:683-720 with D3; power_flow.py:105-121 with D1)
  {
    const int* inj_ptr = simg + lay.o_inj_ptr;
    const int* inj_idx = simg + lay.o_inj_idx;
    if (wide_group<LANES>()) {
      // CTA-wide groups read the image from global memory: the list bounds and the first source of FOUR positions
      // are fetched together, so a lane waits for two L2 round trips per four positions instead of eight
      for (int k0 = g.lane; k0 < lay.P; k0 += 4 * LANES) {
        int qb[4], qe[4], j0[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int k = k0 + u * LANES;
          const bool in = k < lay.P;
          qb[u] = in ? inj_ptr[k] : 0;
          qe[u] = in ? inj_ptr[k + 1] : 0;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) j0[u] = qb[u] < qe[u] ? inj_idx[qb[u]] : 0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int k = k0 + u * LANES;
          if (k >= lay.P) break;
          double ld = 0.0, gn = 0.0;
          for (int q = qb[u]; q < qe[u]; ++q) {
            const int j = q == qb[u] ? j0[u] : inj_idx[q];
            const double v = g.scr(j);
            if (j < L) ld += v;
            else if (j < L + G) gn += v;
            else if (v > 0.0) gn += v;
            else if (v < 0.0) ld += fabs(v);
          }
          g.set_pspec(k, fma(gn, lay.inv_s_base, -ld * lay.inv_s_base));
        }
      }
    } else
    for (int k = g.lane; k < lay.P; k += LANES) {        // by schedule position: lane k % LANES is the one that reads position k back
      double ld = 0.0, gn = 0.0;
      for (int q = inj_ptr[k]; q < inj_ptr[k + 1]; ++q) {
        int j = inj_idx[q];
        double v = g.scr(j);
        if (j < L) ld += v;
        else if (j < L + G) gn += v;
        else if (v > 0.0) gn += v;
        else if (v < 0.0) ld += fabs(v);
      }
      // write after every lane has read its sources: F_P is not part of the scratch region
      g.set_pspec(k, fma(gn, lay.inv_s_base, -ld * lay.inv_s_base));
    }
  }
  g.sync();
  flat_start(g, lay, simg, dimg);
  SolveStat st;
  run_solver<SOLVER>(g, lay, simg, dimg, cfg, &st);

  // ---- bus state -> observation (grid_env.py:722-731, 753-765), reductions for reward / constraints
  double dev = 0.0, vmax = -INFINITY, vmin = INFINITY;
  int v_hi = 0, v_lo = 0;
  {
    const int* rank = simg + lay.o_rank;
    constexpr int UB = wide_group<LANES>() ? 4 : 1;     // image in global memory: four indices per L2 round trip
    for (int i0 = g.lane; i0 < n; i0 += UB * LANES) {
      int kk[UB];
#pragma unroll
      for (int u = 0; u < UB; ++u) kk[u] = i0 + u * LANES < n ? rank[i0 + u * LANES] : 0;
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        const int i = i0 + u * LANES;
        if (i >= n) break;
        const D2 vv = g.ef(kk[u]);
        double e = vv.x, f = vv.y;
        double vm = sqrt(e * e + f * f);
        ob.put2(2 * i, vm, atan2_bus(f, e));
        dev += fabs(vm - 1.0);
        vmax = max_nan(vmax, vm);
        vmin = min_nan(vmin, vm);
        v_hi |= vm > cfg.v_max;
        v_lo |= vm < cfg.v_min;
      }
    }
  }
  double loss_pu = 0.0;
  int over80 = 0;
  {
    if (wide_group<LANES>()) {
      // image in global memory: branch positions, then records / admittances / ratings, of four lines at a time
      const int* bol = simg + lay.o_branch_of_line;
      const I4* sched = reinterpret_cast<const I4*>(simg + lay.o_sched);
      const D2* gb = reinterpret_cast<const D2*>(dimg + lay.o_gb);
      for (int l0 = g.lane; l0 < m; l0 += 4 * LANES) {
        int pb[4]; I4 tt[4]; D2 yy[4]; double rt[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) pb[u] = l0 + u * LANES < m ? bol[l0 + u * LANES] : -1;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          tt[u].x = tt[u].y = tt[u].z = tt[u].w = 0; yy[u].x = yy[u].y = 0.0; rt[u] = 0.0;
          if (pb[u] >= 0) { tt[u] = sched[pb[u]]; yy[u] = gb[pb[u]]; rt[u] = dimg[lay.o_rating + pb[u]]; }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int li = l0 + u * LANES;
          if (li >= m) break;
          double P, S, ls, rating;
          if (pb[u] >= 0) { branch_flow_rec(g, tt[u], yy[u], &P, &S, &ls); rating = rt[u]; }
          else line_flow(g, lay, simg, dimg, li, &P, &S, &ls, &rating);          // a tie
          loss_pu += ls;
          double pw = P * lay.s_base;
          double loading = rating > 0.0 ? fabs(pw) * rcp_fast(rating) : 0.0;
          ob.put2(o_line + 2 * li, pw, loading);
          over80 += loading > 0.8;
        }
      }
    } else
    for (int li = g.lane; li < m; li += LANES) {
      double P, S, ls, rating;
      line_flow(g, lay, simg, dimg, li, &P, &S, &ls, &rating);
      loss_pu += ls;
      double pw = P * lay.s_base;
      double loading = rating > 0.0 ? fabs(pw) * rcp_fast(rating) : 0.0;     // Line.update_state, base.py:261-264 (|P| / rating)
      ob.put2(o_line + 2 * li, pw, loading);
      over80 += loading > 0.8;
    }
  }
  dev = g.gsum(dev);
  loss_pu = g.gsum(loss_pu);
  over80 = g.gsum(over80);
  vmax = g.gmax_nan(vmax);
  vmin = g.gmin_nan(vmin);
  v_hi = g.gor(v_hi); v_lo = g.gor(v_lo);
  tot_ren = g.gsum(tot_ren); tot_used = g.gsum(tot_used); soc_reward = g.gsum(soc_reward);

  // ---- losses, frequency (grid_env.py:733-751; dynamics.py:260-273)
  const double losses_w = loss_pu * lay.s_base;
  total_losses += losses_w * dt / 3600.0;
  {
    double imb = (tot_ren - lay.load_p_sum - losses_w) / 1e6;
    double df = (imb - 1.0 * (freq - 60.0)) / (2.0 * 5.0 * 60.0);
    freq = clampd(freq + df * dt, 55.0, 65.0);
  }
  // ---- reward (grid_env.py:785-826)
  double reward = 0.0;
  reward -= dev * 10.0;
  reward -= fabs(freq - 60.0) * 20.0;
  reward -= (double)over80 * 50.0;
  reward -= total_losses * 0.1;
  reward += tot_used * 1e-5;
  reward += soc_reward;
  // ---- done / constraints (base.py:140-167; grid_env.py:563-608)
  const int terminated = step >= cfg.episode_length;
  const int f_hi = freq > cfg.f_max, f_lo = freq < cfg.f_min;
  const int anyv = v_hi | v_lo | f_hi | f_lo;
  viol_count += anyv;
  const int truncated = anyv && viol_count > 10;
  if (truncated) reward -= cfg.penalty;
  episode_reward += reward;

  if (g.lane == 0) {
    ob.put(o_freq, freq);
    rec[R_TIME] = t; rec[R_FREQ] = freq; rec[R_WIND] = wind; rec[R_TEMP] = temp; rec[R_CLOUD] = cloud;
    rec[R_TOTAL_LOSSES] = total_losses; rec[R_EPISODE_REWARD] = episode_reward;
    ((uint64_t*)rec)[R_DRAWS] = draw + 1ull;
    ((int32_t*)(rec + R_COUNTS))[0] = step;
    ((int32_t*)(rec + R_COUNTS))[1] = viol_count;
    if (o.reward) o.reward[env] = reward;
    if (o.terminated) o.terminated[env] = (uint8_t)terminated;
    if (o.truncated) o.truncated[env] = (uint8_t)truncated;
    if (o.error) o.error[env] = 0;
    if (o.converged) o.converged[env] = (uint8_t)st.converged;
    if (o.iterations) o.iterations[env] = st.iterations;
    if (o.max_voltage) o.max_voltage[env] = vmax;
    if (o.min_voltage) o.min_voltage[env] = vmin;
    if (o.losses) o.losses[env] = losses_w;
    if (o.max_mismatch) o.max_mismatch[env] = st.max_mismatch;
    if (o.violations) {
      o.violations[env * 4 + 0] = (uint8_t)v_hi; o.violations[env * 4 + 1] = (uint8_t)v_lo;
      o.violations[env * 4 + 2] = (uint8_t)f_hi; o.violations[env * 4 + 3] = (uint8_t)f_lo;
    }
    if (o.violation_count) o.violation_count[env] = viol_count;
    if (o.current_step) o.current_step[env] = step;
    if (o.episode_reward) o.episode_reward[env] = episode_reward;
  }
  g.sync();   // the working set is reused by the group's next instance
}

// GridEnvironment.reset (grid_env.py:360-408): counters to zero, buses at 1.0 / 0, lines idle,
// 60 Hz, batteries at their initial state of charge, one weather update at t = 0, full observation.
template <int LANES>
GFR_HD void reset_instance(const Lanes<LANES>& g, const Layout& lay, const int* simg,
                           const double* dimg, const EnvCfg& cfg, long long env, double* state,
                           void* obs, int obs_f32, const double* load_pq, const double* bat_soc0,
                           const uint64_t* seeds, const double* noise, double start_time,
                           bool construct, long long env_id_offset) {
  const int n = lay.n, m = lay.m, L = lay.L, G = lay.G, Bt = lay.Bt, D = lay.D;
  double* rec = state + env * lay.R;
  const ObsRow ob = obs_row(obs, obs, obs_f32, env, D);
  const int o_line = 2 * n, o_freq = 2 * n + 2 * m, o_load = o_freq + 1, o_gen = o_load + 2 * L,
            o_bat = o_gen + G;
  uint64_t seed = seeds ? seeds[env] : ((const uint64_t*)rec)[R_SEED];
  uint64_t draw = (seeds || construct) ? 0ull : ((const uint64_t*)rec)[R_DRAWS];
  // wind / temperature / cloud survive a reset (grid_env.py:673-681); construction sets 5 / 25 / 0.3
  double wind = construct ? 5.0 : rec[R_WIND], temp = construct ? 25.0 : rec[R_TEMP],
         cloud = construct ? 0.3 : rec[R_CLOUD];
  // construction keys instance i with its GLOBAL id, so unseeded shards of one job draw different streams
  if (construct && !seeds) seed = (uint64_t)(env_id_offset + env);
  const bool draws = cfg.weather_variation && !construct;
  if (draws) {
    double u, z1, z2, z3, dummy;
    if (noise) { const double* nz = noise + env * 4; u = nz[0]; z1 = nz[1]; z2 = nz[2]; z3 = nz[3]; }
    else {
      noise_block(seed, draw, 0u, &u, &dummy);
      noise_block(seed, draw, 1u, &z1, &z2);
      noise_block(seed, draw, 2u, &z3, &dummy);
    }
    // the reference resets its clock to 0 before this update (grid_env.py:372, :402): the reset observation is
    // taken at t = 0 whatever `start_time` (a harness extension: the time of day the FIRST STEP starts from) says
    update_weather(hour_of(0.0), u, z1, z2, z3, &wind, &temp, &cloud);
  }
  g.sync();   // every lane has read the record (weather, seed, draw counter) before lane 0 rewrites it
  for (int i = g.lane; i < n; i += LANES) { ob.put(2 * i, 1.0); ob.put(2 * i + 1, 0.0); }
  for (int li = g.lane; li < m; li += LANES) { ob.put(o_line + 2 * li, 0.0); ob.put(o_line + 2 * li + 1, 0.0); }
  for (int l = g.lane; l < 2 * L; l += LANES) ob.put(o_load + l, load_pq[l]);
  for (int gi = g.lane; gi < G; gi += LANES)
    ob.put(o_gen + gi, renewable_power(lay, simg, dimg, gi, hour_of(0.0), wind, temp, cloud));
  for (int b = g.lane; b < Bt; b += LANES) {
    rec[R_BAT + b] = bat_soc0[b]; rec[R_BAT + Bt + b] = 0.0;
    ob.put(o_bat + 2 * b, bat_soc0[b]); ob.put(o_bat + 2 * b + 1, 0.0);
  }
  if (g.lane == 0) {
    ob.put(o_freq, 60.0);
    rec[R_TIME] = start_time; rec[R_FREQ] = 60.0; rec[R_WIND] = wind; rec[R_TEMP] = temp;
    rec[R_CLOUD] = cloud; rec[R_TOTAL_LOSSES] = 0.0; rec[R_EPISODE_REWARD] = 0.0;
    ((uint64_t*)rec)[R_SEED] = seed;
    ((uint64_t*)rec)[R_DRAWS] = draws ? draw + 1ull : draw;
    ((int32_t*)(rec + R_COUNTS))[0] = 0;
    ((int32_t*)(rec + R_COUNTS))[1] = 0;
  }
}

}  // namespace gfr
