// gfr_b200.cu - kernels (sm_100a) and the C ABI declared in include/gfr_b200.h.
//
// Launch shape: persistent CTAs; a group of LANES threads takes instance after instance
// (stride gridDim * groups-per-CTA).  Warp-sized groups never meet a CTA-wide barrier after the
// prologue, so an instance whose solve converges early frees its group early; CTA-wide groups
// (LANES > 32, one instance per CTA) synchronise with __syncthreads.  The prologue stages the
// compiled feeder ("image") into shared memory with ONE bulk async copy (TMA, cp.async.bulk ->
// SASS UBLKCP) completed on an mbarrier, unless the plan reads it from global memory.
// plan_launch() picks instance slots per CTA and CTAs per SM with the occupancy API.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/gfr_b200.h"
#include "gfr_device.cuh"
#include "gfr_dense.cuh"
#include "gfr_image.hpp"

using namespace gfr;

// ----------------------------------------------------------------------------- device side

namespace {

constexpr int kSmemHeader = 16;   // the mbarrier, keeps the image 16-byte aligned
// threads per CTA the kernels are compiled for (sets their register budget: 65536 / threads).
// Measured, no gain: 768 threads (80 registers) for small groups (IEEE-34 237 M -> 230 M env-steps/s).
constexpr int kMaxThreads = 512;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// One elected thread issues the bulk copy global -> shared; everyone waits on the mbarrier.
__device__ __forceinline__ void stage_image(unsigned char* smem, const void* img, int bytes) {
  const uint32_t bar = smem_u32(smem);
  const uint32_t dst = smem_u32(smem + kSmemHeader);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(1) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
        "l"(img), "r"(bytes), "r"(bar)
        : "memory");
  }
  uint32_t ok = 0;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(0)
        : "memory");
  } while (!ok);
}

constexpr int kRedBytes = 128;    // cross-warp reduction scratch of a CTA-wide group (16 doubles)

// Shared memory of a CTA: [mbarrier 16 B][feeder image, if staged][reduction scratch, if LANES > 32][slots]
template <int LANES, int SOLVER, bool SPEC_Q = false>
__device__ __forceinline__ typename GroupOf<LANES, SOLVER>::type
make_group(const Layout& lay, unsigned char* work, int slot_bytes, D2* mscratch, double* p_local) {
  typename GroupOf<LANES, SOLVER>::type g;
  g.lane = threadIdx.x % LANES;
  g.mask = (LANES >= 32) ? 0xffffffffu
                         : (((1u << (LANES & 31)) - 1u) << (((threadIdx.x & 31) / LANES) * LANES));
  g.red = reinterpret_cast<double*>(work);
  if (LANES > 32) work += kRedBytes;
  const int slot = threadIdx.x / LANES;
  const int E = blockDim.x / LANES;
  D2* mg = mscratch ? mscratch + ((size_t)blockIdx.x * E + slot) * (newton_scratch_doubles(lay.P, SPEC_Q) / 2) : nullptr;
  bind_slot<LANES, SPEC_Q>(g, work + (size_t)slot * slot_bytes, lay, mg, p_local);
  return g;
}

// IMG_SMEM: the feeder image is staged into shared memory (small / medium feeders); otherwise it is
// read through L1 / L2 from global memory and all of shared memory goes to the working sets.
template <int LANES, int SOLVER, bool IMG_SMEM>
__global__ void __launch_bounds__(kMaxThreads)
step_kernel(const Layout lay, const EnvCfg cfg, const void* __restrict__ img, const int slot_bytes,
            D2* __restrict__ mscratch, double* __restrict__ state, void* __restrict__ obs,
            const void* obs_prev, const int obs_f32,
            const double* __restrict__ actions, const double* __restrict__ noise, const StepOut o,
            const long long B) {
  extern __shared__ __align__(16) unsigned char smem[];
  if (IMG_SMEM) stage_image(smem, img, lay.img_bytes);
  const int* simg = IMG_SMEM ? (const int*)(smem + kSmemHeader) : (const int*)img;
  const double* dimg = IMG_SMEM ? (const double*)(smem + kSmemHeader) : (const double*)img;
  double p_local[LANES == 1 && SOLVER != SOLVER_NEWTON ? SWEEP_P_LOCAL_MAX : 1];
  auto g = make_group<LANES, SOLVER>(lay, smem + kSmemHeader + (IMG_SMEM ? lay.img_bytes : 0),
                                     slot_bytes, mscratch, p_local);
  const int E = blockDim.x / LANES;
  for (long long env = (long long)blockIdx.x * E + threadIdx.x / LANES; env < B; env += (long long)gridDim.x * E)
    step_instance<LANES, SOLVER>(g, lay, simg, dimg, cfg, env, state, obs, obs_prev, obs_f32, actions, noise, o);
}

template <int LANES, int SOLVER, bool IMG_SMEM>
__global__ void __launch_bounds__(kMaxThreads)
solve_kernel(const Layout lay, const EnvCfg cfg, const void* __restrict__ img, const int slot_bytes,
             D2* __restrict__ mscratch, const double* __restrict__ p_inj, const SolOut o, const long long B) {
  extern __shared__ __align__(16) unsigned char smem[];
  if (IMG_SMEM) stage_image(smem, img, lay.img_bytes);
  const int* simg = IMG_SMEM ? (const int*)(smem + kSmemHeader) : (const int*)img;
  const double* dimg = IMG_SMEM ? (const double*)(smem + kSmemHeader) : (const double*)img;
  double p_local[LANES == 1 && SOLVER != SOLVER_NEWTON ? SWEEP_P_LOCAL_MAX : 1];
  auto g = make_group<LANES, SOLVER>(lay, smem + kSmemHeader + (IMG_SMEM ? lay.img_bytes : 0),
                                     slot_bytes, mscratch, p_local);
  const int E = blockDim.x / LANES;
  for (long long env = (long long)blockIdx.x * E + threadIdx.x / LANES; env < B; env += (long long)gridDim.x * E)
    solve_instance<LANES, SOLVER>(g, lay, simg, dimg, cfg, env, p_inj, o);
}

// solve_kernel with specified Q at the PQ buses (q_inj [B, n]).  A kernel of its own, so that solve_kernel, which
// P-only callers run, keeps its machine code: the Newton scratch holds (P, Q) pairs, the sweep slot 48 B per bus
template <int LANES, int SOLVER, bool IMG_SMEM>
__global__ void __launch_bounds__(kMaxThreads)
solve_pq_kernel(const Layout lay, const EnvCfg cfg, const void* __restrict__ img, const int slot_bytes,
                D2* __restrict__ mscratch, const double* __restrict__ p_inj, const double* __restrict__ q_inj,
                const SolOut o, const long long B) {
  extern __shared__ __align__(16) unsigned char smem[];
  if (IMG_SMEM) stage_image(smem, img, lay.img_bytes);
  const int* simg = IMG_SMEM ? (const int*)(smem + kSmemHeader) : (const int*)img;
  const double* dimg = IMG_SMEM ? (const double*)(smem + kSmemHeader) : (const double*)img;
  auto g = make_group<LANES, SOLVER, true>(lay, smem + kSmemHeader + (IMG_SMEM ? lay.img_bytes : 0),
                                           slot_bytes, mscratch, nullptr);
  const int E = blockDim.x / LANES;
  for (long long env = (long long)blockIdx.x * E + threadIdx.x / LANES; env < B; env += (long long)gridDim.x * E)
    solve_instance<LANES, SOLVER, true>(g, lay, simg, dimg, cfg, env, p_inj, o, q_inj);
}

// reset: 4 lanes per instance, image read through L2 (touched once per instance)
__global__ void __launch_bounds__(128)
reset_kernel(const Layout lay, const EnvCfg cfg, const void* __restrict__ img,
             double* __restrict__ state, void* __restrict__ obs, const int obs_f32,
             const double* __restrict__ load_pq, const double* __restrict__ bat_soc0,
             const uint64_t* __restrict__ seeds, const uint8_t* __restrict__ mask,
             const double* __restrict__ noise, const double start_time, const int construct,
             const long long env_id_offset, const long long B) {
  constexpr int LANES = 4;
  Lanes<LANES> g;
  g.red = nullptr;
  g.lane = threadIdx.x % LANES;
  g.mask = ((1u << LANES) - 1u) << (((threadIdx.x & 31) / LANES) * LANES);
  const int* simg = (const int*)img;
  const double* dimg = (const double*)img;
  const int E = blockDim.x / LANES;
  for (long long env = (long long)blockIdx.x * E + threadIdx.x / LANES; env < B; env += (long long)gridDim.x * E) {
    if (mask && !mask[env]) continue;
    reset_instance<LANES>(g, lay, simg, dimg, cfg, env, state, obs, obs_f32, load_pq, bat_soc0, seeds, noise,
                          start_time, construct != 0, env_id_offset);
  }
}

// the observation the library holds (fp64) into a buffer the caller binds (fp64 or fp32)
__global__ void obs_convert_kernel(const double* __restrict__ src, void* __restrict__ dst, const int f32, const long long count) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    if (f32) reinterpret_cast<float*>(dst)[i] = (float)src[i];
    else reinterpret_cast<double*>(dst)[i] = src[i];
  }
}

// FP64 pipe microbenchmark: 8 independent DFMA chains per thread (the roofline denominator that
// MEASURED_PEAKS.json does not carry; SURVEY 8d)
// The info rows of the instances a reset touched (grid_env.py:360-408: counters and episode sums to zero, voltages
// at 1.0): one launch instead of one masked fill per output array
__global__ void __launch_bounds__(256) reset_outputs_kernel(const StepOut o, const uint8_t* __restrict__ mask,
                                                            const long long B) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < B; i += (long long)gridDim.x * blockDim.x) {
    if (mask && !mask[i]) continue;
    if (o.reward) o.reward[i] = 0.0;
    if (o.terminated) o.terminated[i] = 0;
    if (o.truncated) o.truncated[i] = 0;
    if (o.error) o.error[i] = 0;
    if (o.converged) o.converged[i] = 0;
    if (o.iterations) o.iterations[i] = 0;
    if (o.max_voltage) o.max_voltage[i] = 1.0;
    if (o.min_voltage) o.min_voltage[i] = 1.0;
    if (o.losses) o.losses[i] = 0.0;
    if (o.max_mismatch) o.max_mismatch[i] = 0.0;
    if (o.violations) { for (int q = 0; q < 4; ++q) o.violations[i * 4 + q] = 0; }
    if (o.violation_count) o.violation_count[i] = 0;
    if (o.current_step) o.current_step[i] = 0;
    if (o.episode_reward) o.episode_reward[i] = 0.0;
  }
}

__global__ void __launch_bounds__(256) dfma_peak_kernel(double* __restrict__ out, const int iters, const double seed) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1.0, a2 = a0 + 2.0, a3 = a0 + 3.0, a4 = a0 + 4.0, a5 = a0 + 5.0,
         a6 = a0 + 6.0, a7 = a0 + 7.0;
  const double m = 1.0000001, c = 1e-9;
#pragma unroll 4
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

__global__ void noise_fill_kernel(const long long B, const int n_slots,
                                  const uint64_t* __restrict__ seeds,
                                  const uint64_t* __restrict__ draws, double* __restrict__ out) {
  const long long total = B * (long long)n_slots;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long env = i / n_slots;
    const int s = (int)(i - env * n_slots);
    out[i] = noise_slot(seeds[env], draws[env], s);
  }
}

}  // namespace

// ----------------------------------------------------------------------------- host side

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return GFR_E_CUDA;
}
#define GFR_CUDA(call)                                     \
  do {                                                     \
    cudaError_t e_ = (call);                               \
    if (e_ != cudaSuccess) return cuda_fail(e_, #call);    \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    cur = dev;
  }
  ~DeviceGuard() { if (ok && prev >= 0 && prev != cur) cudaSetDevice(prev); }
  int cur = -1;
};
// what an entry point that needs the device returns when DeviceGuard could not switch to it
int no_device() { return fail(GFR_E_CUDA, "no usable CUDA device (this library has no CPU fallback)"); }

}  // namespace

// one compiled image per (solver, lanes) a feeder has been asked to run on, built on first use
struct ImageDev {
  Layout lay{};
  void* d_img = nullptr;
};

struct gfr_feeder {
  int device = 0;
  int sm_count = 0;
  int smem_optin = 0;
  int smem_per_sm = 0;
  Layout lay{};                  // sizes only (n, L, G, Bt, A, D, R, ...): offsets belong to an image
  bool has_pv = false;
  int lanes_hint = 0;            // lane count the level schedule was capped for (0: not said)
  int center_depth = 0;          // levels of the tree rooted at its center, uncapped
  DescCopy desc;                 // the description, kept to build further images
  mutable std::map<int, ImageDev> images;   // key = solver * 1024 + lanes
  double* d_load_pq = nullptr;   // [2L] static active / reactive power (observation)
  double* d_bat_soc0 = nullptr;  // [Bt]
};

struct gfr_env {
  const gfr_feeder* f = nullptr;
  const ImageDev* img = nullptr;
  long long B = 0;
  EnvCfg cfg{};
  int solver = GFR_SOLVER_NEWTON;
  int lanes = 0, threads = 0, grid = 0;
  size_t smem = 0;
  const void* fn = nullptr;
  double* d_state = nullptr;
  void* d_obs = nullptr;         // the buffer holding the latest observation
  void* d_obs_alt = nullptr;     // the other one of two alternating caller-owned buffers (nullptr: one buffer)
  int obs_f32 = 0;               // caller-bound fp32 observation buffers
  D2* d_mscratch = nullptr;    // Newton: D^-1 U, D^-1 r, specified injections of every resident instance slot (L2 resident)
  int slot_bytes = 0;
  bool obs_external = false;   // bound by gfr_env_bind_obs: caller-owned
  long long env_id_offset = 0; // global id of instance 0 (keys the construction-time Philox streams)
};

struct gfr_network {
  int device = 0;
  int sm_count = 0;
  int smem_optin = 0;
  NetDev nd{};
  void* d_ints = nullptr;       // one allocation each: the int arrays, the double arrays
  void* d_dbls = nullptr;
};

namespace {

struct LaunchPlan { int lanes, threads, grid; size_t smem; int ctas_per_sm; int slot_bytes; size_t mscratch_bytes; bool img_smem; };

// which kernel a launch plan is for: the environment step, the solve, the solve with specified Q
enum KernelKind { K_STEP, K_SOLVE, K_SOLVE_PQ };

// the image of a feeder for one (solver, lanes): built and uploaded on first use
int image_for(const gfr_feeder* f, int solver, int lanes, const ImageDev** out) {
  const int key = solver * 1024 + lanes;
  auto it = f->images.find(key);
  if (it != f->images.end()) { *out = &it->second; return GFR_OK; }
  FeederImage fi;
  std::string complaint = build_feeder_image(&f->desc.d, lanes, solver, &fi);
  if (!complaint.empty()) return fail(GFR_E_ARG, complaint);
  ImageDev dev;
  dev.lay = fi.lay;
  GFR_CUDA(cudaMalloc(&dev.d_img, fi.img.size()));
  cudaError_t ce = cudaMemcpy(dev.d_img, fi.img.data(), fi.img.size(), cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) { cudaFree(dev.d_img); return cuda_fail(ce, "cudaMemcpy(image)"); }
  auto ins = f->images.emplace(key, dev);
  *out = &ins.first->second;
  return GFR_OK;
}

// shared memory of one instance slot; 0 if the scratch it doubles as cannot hold the sources
size_t slot_bytes(const Layout& lay, int solver, int lanes, int kind) {
  const bool spec_q = kind == K_SOLVE_PQ;
  return solver == GFR_SOLVER_NEWTON ? newton_slot_bytes(lay.n, lay.n_pool, lay.n_src)
                                     : sweep_slot_bytes(lay.n, lay.n_src, !spec_q && sweep_p_local(lanes, lay.n), lay.n_tie, spec_q);
}

// Threads cooperating on one instance when the caller does not say: THE rule (exported as gfr_auto_lanes; the
// Python side calls it instead of keeping a copy).  Thresholds from measurements on B200
// (profiles/r01_tune_lanes_newton_v7.txt, profiles/r01_bench_all_configs_v11.txt): a few lanes for the smallest
// feeders, part of a warp up to a few hundred buses, one CTA per instance (feeder image read from global memory)
// beyond.  `depth` = levels of the center-rooted tree (0 = unknown): a small feeder with fewer than four buses per
// level (IEEE-13: 13 / 4, IEEE-34: 34 / 12) keeps only two Newton lanes busy (IEEE-13 510 M -> 566 M, IEEE-34
// 250 M -> 271 M env-steps/s; a bushier 30-bus random tree, 30 / 7, is faster on four).
int auto_lanes_rule(int n, int solver, int depth) {
  if (n <= 45 && solver != GFR_SOLVER_SWEEP && depth > 0 && n < 4 * depth) return 2;
  if (n <= 20) return solver == GFR_SOLVER_SWEEP ? 1 : 4;
  if (n <= 45) return 4;
  if (solver == GFR_SOLVER_SWEEP) {
    if (n <= 90) return 8;
    if (n <= 160) return 16;
  } else {
    if (n <= 160) return 8;
    if (n <= 250) return 16;
  }
  if (n <= 400) return 32;
  if (n <= 1500) return 64;
  return 128;                      // one CTA per instance
}

// The step, solve or Q solve kernel of one (lanes, image placement) out of the lane list L it is compiled for: 1 - 32
// lanes with the image in shared memory, 32 - 256 without it; nullptr for any other lane count
template <int SOLVER, bool IMG_SMEM, int... L>
const void* kernel_in(int kind, int lanes) {
  const void* fn = nullptr;
  auto pick = [&](int l, const void* step_k, const void* solve_k, const void* solve_pq_k) {
    if (lanes == l) fn = kind == K_STEP ? step_k : kind == K_SOLVE ? solve_k : solve_pq_k;
  };
  (pick(L, (const void*)step_kernel<L, SOLVER, IMG_SMEM>, (const void*)solve_kernel<L, SOLVER, IMG_SMEM>,
        (const void*)solve_pq_kernel<L, SOLVER, IMG_SMEM>), ...);
  return fn;
}
template <int SOLVER>
const void* kernel_of(int kind, int lanes, bool img_smem) {
  return img_smem ? kernel_in<SOLVER, true, 1, 2, 4, 8, 16, 32>(kind, lanes)
                  : kernel_in<SOLVER, false, 32, 64, 128, 256>(kind, lanes);
}
const void* kernel_fn(int kind, int solver, int lanes, bool img_smem, bool ties) {
  if (solver == GFR_SOLVER_NEWTON) return kernel_of<SOLVER_NEWTON>(kind, lanes, img_smem);
  return ties ? kernel_of<SOLVER_SWEEP_TIES>(kind, lanes, img_smem) : kernel_of<SOLVER_SWEEP>(kind, lanes, img_smem);
}

// One candidate split of an SM: `c` CTAs of E instance slots each.
struct PlanTry { long long resident = 0; LaunchPlan plan{}; };

PlanTry plan_mode(const gfr_feeder* f, const Layout& lay, const void* fn, int lanes, bool img_smem, size_t per_env, long long B) {
  PlanTry best;
  if (!fn) return best;
  if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, f->smem_optin) != cudaSuccess) {
    cudaGetLastError();
    return best;
  }
  const size_t fixed = kSmemHeader + (img_smem ? (size_t)lay.img_bytes : 0) + (lanes > 32 ? kRedBytes : 0);
  const size_t sm_total = (size_t)f->smem_per_sm;
  const int gran = lanes >= 32 ? 1 : 32 / lanes;         // whole warps
  // pass 0: whole warps only; pass 1 (only if nothing fits): a partial warp
  for (int pass = 0; pass < 2 && !best.resident; ++pass) {
    for (int c = 1; c <= 16; ++c) {
      const size_t share = sm_total / c;
      if (share < fixed + per_env + 1024) break;
      long long E = (long long)((share - 1024 - fixed) / per_env);
      if (lanes > 32) E = 1;                              // one CTA per instance
      if (E * lanes > kMaxThreads) E = kMaxThreads / lanes;
      if (pass == 0) E -= E % gran;                        // (a partial last warp was measured: no gain)
      if (E < 1) continue;
      const int threads = (int)(E * lanes);
      const size_t smem = fixed + per_env * (size_t)E;
      if (smem > (size_t)f->smem_optin) continue;
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, threads, smem) != cudaSuccess) { cudaGetLastError(); continue; }
      if (nb > c && lanes <= 32) nb = c;
      const long long resident = (long long)nb * E;
      // more resident instances win.  On a tie: a short launch (few waves) takes more, smaller CTAs,
      // which even out its last wave; a long one takes fewer, so that fewer copies of the image are staged
      const bool short_launch = B < 8 * (long long)f->sm_count * (resident > 0 ? resident : 1);
      const bool tie = resident == best.resident && resident > 0 &&
                       (short_launch ? nb > best.plan.ctas_per_sm : nb < best.plan.ctas_per_sm);
      if (resident > best.resident || tie) {
        best.resident = resident;
        best.plan.lanes = lanes; best.plan.threads = threads; best.plan.smem = smem; best.plan.ctas_per_sm = nb;
        best.plan.img_smem = img_smem;
      }
      if (lanes > 32) break;                               // E is fixed: the occupancy API said how many CTAs fit
    }
  }
  return best;
}

// Instance slots per CTA and CTAs per SM: the split of an SM's shared memory that keeps the most
// instances resident, checked against the kernel's real register use through the occupancy API.
// Small and medium feeders stage one copy of the feeder image per CTA; when that leaves fewer than
// four instances resident (or the group is CTA-wide) the image is read from global memory instead.
int plan_launch(const gfr_feeder* f, int kind, int solver, int lanes, long long B, LaunchPlan* out,
                const void** fn_out, const ImageDev** img_out) {
  // the lane count the description's level schedule was capped for, else the rule
  if (lanes == 0) lanes = f->lanes_hint > 0 ? f->lanes_hint : auto_lanes_rule(f->lay.n, solver, f->center_depth);
  if (lanes != 1 && lanes != 2 && lanes != 4 && lanes != 8 && lanes != 16 && lanes != 32 && lanes != 64 &&
      lanes != 128 && lanes != 256)
    return fail(GFR_E_ARG, "lanes must be 0 (auto), 1, 2, 4, 8, 16, 32 (part of a warp) or 64, 128, 256 (one CTA per instance)");
  const ImageDev* im = nullptr;
  if (int rc = image_for(f, solver, lanes, &im)) return rc;
  const Layout& lay = im->lay;
  *img_out = im;
  const size_t per_env = slot_bytes(lay, solver, lanes, kind);
  if (!per_env)
    return fail(GFR_E_LIMIT, "more loads + generators + batteries than the solver's working set can stage "
                             "(sweep: 2 per bus on average)");
  PlanTry best;
  if (lanes <= 32) best = plan_mode(f, lay, kernel_fn(kind, solver, lanes, true, lay.n_tie > 0), lanes, true, per_env, B);
  if (lanes > 32 || (lanes == 32 && best.resident < 4)) {
    PlanTry alt = plan_mode(f, lay, kernel_fn(kind, solver, lanes, false, lay.n_tie > 0), lanes, false, per_env, B);
    if (alt.resident > best.resident) best = alt;
  }
  if (!best.resident)
    return fail(GFR_E_LIMIT, "one instance's working set (plus the feeder image) exceeds the shared memory of an SM");
  LaunchPlan plan = best.plan;
  long long E = plan.threads / lanes;
  if (lanes <= 32) {
    // A short launch (a few waves of resident instances) is evened out: the same number of waves, every CTA of
    // every wave with the same number of instances - fewer slots per CTA instead of a nearly empty last wave
    // (IEEE-13, 65 536 instances: 352 slots per SM made waves of 352 + 91; now 2 x 224), and a batch smaller than
    // one wave spreads over all SMs instead of filling the first CTAs.
    const long long ctas = (long long)f->sm_count * plan.ctas_per_sm;
    const long long waves = (B + ctas * E - 1) / (ctas * E);
    if (waves <= 8) {
      const int gran = lanes >= 32 ? 1 : 32 / lanes;
      long long need = (B + waves * ctas - 1) / (waves * ctas);
      need = (need + gran - 1) / gran * gran;
      if (need >= 1 && need < E) {
        plan.smem -= per_env * (size_t)(E - need);
        E = need;
        plan.threads = (int)(E * lanes);
      }
    }
  }
  long long tiles = (B + E - 1) / E;
  long long grid = (long long)f->sm_count * plan.ctas_per_sm;
  if (grid > tiles) grid = tiles;
  if (lanes > 32 && grid > 0) {
    // one instance per CTA: the same number of rounds for every CTA (2 048 instances on 8 x 148 resident CTAs made
    // 864 CTAs with two instances and 320 with one; 1 024 with two each leave every SM a CTA less to interleave)
    const long long rounds = (tiles + grid - 1) / grid;
    if (rounds <= 8) grid = (tiles + rounds - 1) / rounds;
  }
  if (grid < 1) grid = 1;
  plan.grid = (int)grid;
  plan.slot_bytes = (int)per_env;
  // Newton spills D^-1 U (32 B per bus) of every resident instance slot to global memory
  plan.mscratch_bytes = solver == GFR_SOLVER_NEWTON ? (size_t)grid * E * newton_scratch_doubles(lay.P, kind == K_SOLVE_PQ) * 8 : 0;
  *out = plan;
  *fn_out = kernel_fn(kind, solver, lanes, plan.img_smem, lay.n_tie > 0);
  return GFR_OK;
}

int launch_step(const gfr_env* e, const double* actions, const double* noise, const StepOut& o,
                cudaStream_t s) {
  const void* img = e->img->d_img;
  double* state = e->d_state;
  // two alternating buffers: this step writes the one that does not hold the latest observation
  const void* obs_prev = e->d_obs;
  void* obs = e->d_obs_alt ? e->d_obs_alt : e->d_obs;
  int f32 = e->obs_f32;
  long long B = e->B;
  int slot = e->slot_bytes;
  D2* ms = e->d_mscratch;
  void* args[] = {(void*)&e->img->lay, (void*)&e->cfg, (void*)&img, (void*)&slot, (void*)&ms, (void*)&state,
                  (void*)&obs, (void*)&obs_prev, (void*)&f32, (void*)&actions, (void*)&noise, (void*)&o, (void*)&B};
  GFR_CUDA(cudaLaunchKernel(e->fn, dim3(e->grid), dim3(e->threads), args, e->smem, s));
  g_launches.fetch_add(1);
  if (e->d_obs_alt) std::swap(const_cast<gfr_env*>(e)->d_obs, const_cast<gfr_env*>(e)->d_obs_alt);
  return GFR_OK;
}

// solve_kernel, or solve_pq_kernel when q_inj is given
int launch_solve(const ImageDev* im, const LaunchPlan& p, const void* fn, const EnvCfg& cfg,
                 const double* p_inj, const double* q_inj, const SolOut& o, long long B, cudaStream_t s) {
  const void* img = im->d_img;
  int slot = p.slot_bytes;
  D2* ms = nullptr;
  if (p.mscratch_bytes) GFR_CUDA(cudaMallocAsync((void**)&ms, p.mscratch_bytes, s));   // stream-ordered scratch
  void* args[] = {(void*)&im->lay, (void*)&cfg, (void*)&img, (void*)&slot, (void*)&ms, (void*)&p_inj, (void*)&o,
                  (void*)&B};
  void* args_pq[] = {(void*)&im->lay, (void*)&cfg, (void*)&img, (void*)&slot, (void*)&ms, (void*)&p_inj,
                     (void*)&q_inj, (void*)&o, (void*)&B};
  cudaError_t le = cudaLaunchKernel(fn, dim3(p.grid), dim3(p.threads), q_inj ? args_pq : args, p.smem, s);
  if (ms) cudaFreeAsync(ms, s);
  if (le != cudaSuccess) return cuda_fail(le, "cudaLaunchKernel(solve)");
  g_launches.fetch_add(1);
  return GFR_OK;
}

// the stopping rule of every solve
int check_stopping(const gfr_solver_cfg* c) {
  if (c->max_iterations < 1) return fail(GFR_E_ARG, "max_iterations must be >= 1");
  if (!(c->tolerance > 0.0)) return fail(GFR_E_ARG, "tolerance must be > 0");
  return GFR_OK;
}

int check_solver_cfg(const gfr_feeder* f, const gfr_solver_cfg* c) {
  if (c->solver != GFR_SOLVER_SWEEP && c->solver != GFR_SOLVER_NEWTON)
    return fail(GFR_E_ARG, "solver must be GFR_SOLVER_SWEEP or GFR_SOLVER_NEWTON");
  if (int rc = check_stopping(c)) return rc;
  if (c->solver == GFR_SOLVER_SWEEP && f->has_pv)
    return fail(GFR_E_ARG, "the sweep solver handles slack + PQ buses only; use GFR_SOLVER_NEWTON for PV buses");
  return GFR_OK;
}

}  // namespace

extern "C" {

int gfr_abi_version(void) { return GFR_ABI_VERSION; }
const char* gfr_last_error(void) { return g_err.c_str(); }
int64_t gfr_launch_count(void) { return g_launches.load(); }
int gfr_auto_lanes(int n_bus, int solver, int depth) { return auto_lanes_rule(n_bus, solver, depth); }

int gfr_feeder_create(const gfr_feeder_desc* d, int device, gfr_feeder** out) {
  if (!d || !out) return fail(GFR_E_ARG, "null argument");
  *out = nullptr;
  // the description is checked (and a first image built on the host) before a device is asked for
  FeederImage fi;
  {
    const int lanes0 = d->lanes_hint > 0 && d->lanes_hint <= 256 ? d->lanes_hint : 1;
    // (a feeder with ties only has sweep images)
    std::string complaint = build_feeder_image(d, lanes0, d->n_tie > 0 ? GFR_SOLVER_SWEEP : GFR_SOLVER_NEWTON, &fi);
    if (!complaint.empty()) return fail(GFR_E_ARG, complaint);
  }
  DeviceGuard guard(device);
  if (!guard.ok) return no_device();
  cudaDeviceProp prop;
  GFR_CUDA(cudaGetDeviceProperties(&prop, device));
  auto* f = new gfr_feeder();
  f->device = device;
  f->sm_count = prop.multiProcessorCount;
  f->smem_optin = (int)prop.sharedMemPerBlockOptin;
  f->smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
  f->lay = fi.lay;
  f->has_pv = fi.has_pv;
  f->lanes_hint = d->lanes_hint;
  f->center_depth = fi.center_depth;
  f->desc.assign(d);
  const int Bt = f->lay.Bt;
  const std::vector<double>& load_pq = fi.load_pq;
  cudaError_t e2 = cudaMalloc((void**)&f->d_load_pq, load_pq.size() * 8);
  cudaError_t e3 = cudaMalloc((void**)&f->d_bat_soc0, ((size_t)Bt + 1) * 8);
  if (e2 != cudaSuccess || e3 != cudaSuccess) {
    gfr_feeder_destroy(f);
    return cuda_fail(e2 != cudaSuccess ? e2 : e3, "cudaMalloc(feeder)");
  }
  cudaError_t c2 = cudaMemcpy(f->d_load_pq, load_pq.data(), load_pq.size() * 8, cudaMemcpyHostToDevice);
  cudaError_t c3 = Bt ? cudaMemcpy(f->d_bat_soc0, d->bat_soc0, (size_t)Bt * 8, cudaMemcpyHostToDevice) : cudaSuccess;
  if (c2 != cudaSuccess || c3 != cudaSuccess) {
    gfr_feeder_destroy(f);
    return cuda_fail(c2 != cudaSuccess ? c2 : c3, "cudaMemcpy(feeder)");
  }
  *out = f;
  return GFR_OK;
}

void gfr_feeder_destroy(gfr_feeder* f) {
  if (!f) return;
  DeviceGuard guard(f->device);
  for (auto& kv : f->images) cudaFree(kv.second.d_img);
  cudaFree(f->d_load_pq);
  cudaFree(f->d_bat_soc0);
  delete f;
}

static int fill_env_cfg(const gfr_feeder* f, const gfr_env_cfg* c, EnvCfg* out) {
  if (int rc = check_solver_cfg(f, &c->solver)) return rc;
  if (!(c->timestep > 0.0)) return fail(GFR_E_ARG, "timestep must be > 0");
  if (c->episode_length < 1) return fail(GFR_E_ARG, "episode_length must be >= 1");
  *out = env_cfg_of(c);
  return GFR_OK;
}

static int launch_reset(gfr_env* e, const uint64_t* seeds, const uint8_t* mask, const double* noise,
                        double start_time, int construct, cudaStream_t s) {
  const int threads = 128, per_cta = threads / 4;
  long long grid = (e->B + per_cta - 1) / per_cta;
  const long long cap = (long long)e->f->sm_count * 16;
  if (grid > cap) grid = cap;
  reset_kernel<<<(int)grid, threads, 0, s>>>(e->img->lay, e->cfg, e->img->d_img, e->d_state, e->d_obs, e->obs_f32,
                                            e->f->d_load_pq, e->f->d_bat_soc0, seeds, mask, noise,
                                            start_time, construct, e->env_id_offset, e->B);
  g_launches.fetch_add(1);
  GFR_CUDA(cudaGetLastError());
  return GFR_OK;
}

int gfr_env_create(const gfr_feeder* f, int64_t n_envs, const gfr_env_cfg* cfg, gfr_env** out) {
  if (!f || !cfg || !out) return fail(GFR_E_ARG, "null argument");
  *out = nullptr;
  if (n_envs < 1) return fail(GFR_E_ARG, "n_envs must be >= 1");
  EnvCfg ec;
  if (int rc = fill_env_cfg(f, cfg, &ec)) return rc;
  DeviceGuard guard(f->device);
  if (!guard.ok) return no_device();
  LaunchPlan plan;
  const void* fn = nullptr;
  const ImageDev* im = nullptr;
  if (int rc = plan_launch(f, K_STEP, cfg->solver.solver, cfg->solver.lanes, n_envs, &plan, &fn, &im)) return rc;
  auto* e = new gfr_env();
  e->f = f; e->img = im; e->B = n_envs; e->cfg = ec; e->solver = cfg->solver.solver;
  e->lanes = plan.lanes; e->threads = plan.threads; e->grid = plan.grid; e->smem = plan.smem; e->fn = fn;
  e->slot_bytes = plan.slot_bytes;
  e->env_id_offset = cfg->env_id_offset;
  cudaError_t e1 = cudaMalloc((void**)&e->d_state, (size_t)n_envs * f->lay.R * 8);
  cudaError_t e2 = cudaMalloc((void**)&e->d_obs, (size_t)n_envs * f->lay.D * 8);
  if (e1 == cudaSuccess && e2 == cudaSuccess && plan.mscratch_bytes)
    e2 = cudaMalloc((void**)&e->d_mscratch, plan.mscratch_bytes);
  if (e1 != cudaSuccess || e2 != cudaSuccess) {
    gfr_env_destroy(e);
    return cuda_fail(e1 != cudaSuccess ? e1 : e2, "cudaMalloc(env)");
  }
  if (int rc = launch_reset(e, nullptr, nullptr, nullptr, 0.0, 1, 0)) { gfr_env_destroy(e); return rc; }
  cudaError_t es = cudaStreamSynchronize(0);
  if (es != cudaSuccess) { gfr_env_destroy(e); return cuda_fail(es, "reset at construction"); }
  *out = e;
  return GFR_OK;
}

void gfr_env_destroy(gfr_env* e) {
  if (!e) return;
  DeviceGuard guard(e->f->device);
  cudaFree(e->d_state);
  cudaFree(e->d_mscratch);
  if (!e->obs_external) cudaFree(e->d_obs);
  delete e;
}

int64_t gfr_env_num_envs(const gfr_env* e) { return e ? e->B : 0; }
int gfr_env_obs_dim(const gfr_env* e) { return e ? e->f->lay.D : 0; }
int gfr_env_act_dim(const gfr_env* e) { return e ? e->f->lay.A : 0; }
int gfr_env_noise_dim(const gfr_env* e) { return e ? e->f->lay.n_noise : 0; }
double* gfr_env_obs(gfr_env* e) { return e && !e->obs_f32 ? (double*)e->d_obs : nullptr; }
void* gfr_env_obs_current(gfr_env* e) { return e ? e->d_obs : nullptr; }
int64_t gfr_env_state_bytes(const gfr_env* e) { return e ? (int64_t)e->B * e->f->lay.R * 8 : 0; }

int gfr_env_bind_obs_buffers(gfr_env* e, void* obs_a, void* obs_b, int dtype, void* stream) {
  if (!e || !obs_a) return fail(GFR_E_ARG, "null argument");
  if (dtype != GFR_OBS_F64 && dtype != GFR_OBS_F32) return fail(GFR_E_ARG, "dtype must be GFR_OBS_F64 or GFR_OBS_F32");
  if (obs_a == obs_b) return fail(GFR_E_ARG, "the two observation buffers must differ");
  DeviceGuard guard(e->f->device);
  cudaStream_t s = (cudaStream_t)stream;
  const long long count = (long long)e->B * e->f->lay.D;
  // the observation so far (fp64 if the library still owns it, else the bound type) moves into the new buffers
  void* bufs[2] = {obs_a, obs_b};
  for (int i = 0; i < 2; ++i) {
    if (!bufs[i]) continue;
    if (!e->obs_f32) {
      long long grid = (count + 255) / 256;
      if (grid > (long long)e->f->sm_count * 16) grid = (long long)e->f->sm_count * 16;
      obs_convert_kernel<<<(int)grid, 256, 0, s>>>((const double*)e->d_obs, bufs[i], dtype == GFR_OBS_F32, count);
      g_launches.fetch_add(1);
      GFR_CUDA(cudaGetLastError());
    } else {
      if (dtype != GFR_OBS_F32) return fail(GFR_E_ARG, "an environment bound to fp32 observations stays fp32");
      GFR_CUDA(cudaMemcpyAsync(bufs[i], e->d_obs, (size_t)count * 4, cudaMemcpyDeviceToDevice, s));
    }
  }
  GFR_CUDA(cudaStreamSynchronize(s));
  if (!e->obs_external) cudaFree(e->d_obs);
  e->d_obs = obs_a;
  e->d_obs_alt = obs_b;
  e->obs_f32 = dtype == GFR_OBS_F32;
  e->obs_external = true;
  return GFR_OK;
}

int gfr_env_bind_obs(gfr_env* e, double* obs, void* stream) {
  return gfr_env_bind_obs_buffers(e, obs, nullptr, GFR_OBS_F64, stream);
}

int gfr_env_obs_to_host(gfr_env* e, const void* obs_device, void* host_dst, int32_t col0, int32_t ncols, void* stream) {
  if (!e || !obs_device || !host_dst) return fail(GFR_E_ARG, "null argument");
  const int D = e->f->lay.D;
  if (col0 < 0 || ncols < 1 || col0 + ncols > D) return fail(GFR_E_ARG, "column range outside the observation");
  if (obs_device != e->d_obs && obs_device != e->d_obs_alt) return fail(GFR_E_ARG, "not one of this environment's observation buffers");
  DeviceGuard guard(e->f->device);
  const size_t item = e->obs_f32 ? 4 : 8, pitch = (size_t)D * item;
  // one strided DMA: rows of `ncols` entries, both sides with the full row pitch
  GFR_CUDA(cudaMemcpy2DAsync((char*)host_dst + (size_t)col0 * item, pitch, (const char*)obs_device + (size_t)col0 * item, pitch,
                             (size_t)ncols * item, (size_t)e->B, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return GFR_OK;
}

int gfr_env_launch_info(const gfr_env* e, int32_t* lanes, int32_t* threads, int32_t* grid, int64_t* smem_bytes) {
  if (!e) return fail(GFR_E_ARG, "null env");
  if (lanes) *lanes = e->lanes;
  if (threads) *threads = e->threads;
  if (grid) *grid = e->grid;
  if (smem_bytes) *smem_bytes = (int64_t)e->smem;
  return GFR_OK;
}

int gfr_env_state_get(gfr_env* e, void* dst, void* stream) {
  if (!e || !dst) return fail(GFR_E_ARG, "null argument");
  DeviceGuard guard(e->f->device);
  GFR_CUDA(cudaMemcpyAsync(dst, e->d_state, (size_t)gfr_env_state_bytes(e), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return GFR_OK;
}

int gfr_env_state_set(gfr_env* e, const void* src, void* stream) {
  if (!e || !src) return fail(GFR_E_ARG, "null argument");
  DeviceGuard guard(e->f->device);
  GFR_CUDA(cudaMemcpyAsync(e->d_state, src, (size_t)gfr_env_state_bytes(e), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return GFR_OK;
}

int gfr_env_reset(gfr_env* e, const uint64_t* seeds, const uint8_t* mask, const double* noise,
                  double start_time, void* stream) {
  if (!e) return fail(GFR_E_ARG, "null env");
  if (!(start_time >= 0.0)) return fail(GFR_E_ARG, "start_time must be >= 0");
  DeviceGuard guard(e->f->device);
  return launch_reset(e, seeds, mask, noise, start_time, 0, (cudaStream_t)stream);
}

int gfr_env_step(gfr_env* e, const double* actions, const double* noise, const gfr_step_out* out,
                 void* stream) {
  if (!e || !actions) return fail(GFR_E_ARG, "null argument");
  const StepOut o = out ? *out : StepOut{};
  DeviceGuard guard(e->f->device);
  return launch_step(e, actions, noise, o, (cudaStream_t)stream);
}

int gfr_env_reset_outputs(gfr_env* e, const uint8_t* mask, const gfr_step_out* out, void* stream) {
  if (!e || !out) return fail(GFR_E_ARG, "null argument");
  DeviceGuard guard(e->f->device);
  const long long B = e->B;
  const int threads = 256;
  long long blocks = (B + threads - 1) / threads;
  if (blocks > 4LL * e->f->sm_count) blocks = 4LL * e->f->sm_count;
  reset_outputs_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(*out, mask, B);
  GFR_CUDA(cudaGetLastError());
  g_launches.fetch_add(1);
  return GFR_OK;
}

int gfr_solve(const gfr_feeder* f, int64_t B, const double* p_inj, const gfr_solver_cfg* cfg,
              const gfr_sol_out* out, void* stream) {
  return gfr_solve_pq(f, B, p_inj, nullptr, cfg, out, stream);
}

int gfr_solve_pq(const gfr_feeder* f, int64_t B, const double* p_inj, const double* q_inj, const gfr_solver_cfg* cfg,
                 const gfr_sol_out* out, void* stream) {
  if (!f || !p_inj || !cfg || !out) return fail(GFR_E_ARG, "null argument");
  if (B < 1) return fail(GFR_E_ARG, "B must be >= 1");
  if (int rc = check_solver_cfg(f, cfg)) return rc;
  DeviceGuard guard(f->device);
  if (!guard.ok) return no_device();
  LaunchPlan plan;
  const void* fn = nullptr;
  const ImageDev* im = nullptr;
  if (int rc = plan_launch(f, q_inj ? K_SOLVE_PQ : K_SOLVE, cfg->solver, cfg->lanes, B, &plan, &fn, &im)) return rc;
  return launch_solve(im, plan, fn, env_cfg_of(cfg), p_inj, q_inj, *out, B, (cudaStream_t)stream);
}

int gfr_network_create(const gfr_network_desc* d, int device, gfr_network** out) {
  if (!d || !out) return fail(GFR_E_ARG, "null argument");
  *out = nullptr;
  const int n = d->n_bus, m = d->n_line;
  if (n < 2 || m < 1) return fail(GFR_E_ARG, "a network needs at least two buses and one line");
  if (!(d->s_base > 0.0)) return fail(GFR_E_ARG, "s_base must be > 0");
  if (!d->bus_type || !d->vm_set || !d->line_from || !d->line_to || !d->line_r || !d->line_x || !d->line_rating)
    return fail(GFR_E_ARG, "missing network array");
  // unknowns in the reference's order (power_flow.py:213-295): angles of the non-slack buses, then |V| of the PQ buses
  std::vector<int32_t> col_theta(n, -1), col_vm(n, -1);
  int n_slack = 0, nt = 0;
  for (int i = 0; i < n; ++i) {
    if (d->bus_type[i] != GFR_BUS_SLACK && d->bus_type[i] != GFR_BUS_PV && d->bus_type[i] != GFR_BUS_PQ)
      return fail(GFR_E_ARG, "unknown bus_type");
    if (d->bus_type[i] == GFR_BUS_SLACK) { ++n_slack; continue; }
    col_theta[i] = nt++;
  }
  if (n_slack != 1) return fail(GFR_E_ARG, "exactly one slack bus is required");
  int N = nt;
  for (int i = 0; i < n; ++i) if (d->bus_type[i] == GFR_BUS_PQ) col_vm[i] = N++;
  // Ybus (power_flow.py:48-73): y = 1 / (r + jx), an impedance of magnitude <= 1e-12 is an open line;
  // parallel lines merge into one neighbour entry
  std::vector<double> line_y(2 * (size_t)m), ydiag(2 * (size_t)n, 0.0);
  std::vector<std::map<int, std::pair<double, double>>> nb(n);
  for (int k = 0; k < m; ++k) {
    const int i = d->line_from[k], j = d->line_to[k];
    if (i < 0 || i >= n || j < 0 || j >= n || i == j) return fail(GFR_E_ARG, "line end out of range");
    const double r = d->line_r[k], x = d->line_x[k], z2 = r * r + x * x;
    double g = 0.0, b = 0.0;
    if (std::sqrt(z2) > 1e-12) { g = r / z2; b = -x / z2; }
    if (!(g == g) || !(b == b)) return fail(GFR_E_ARG, "line with NaN impedance");
    line_y[2 * k] = g; line_y[2 * k + 1] = b;
    ydiag[2 * i] += g; ydiag[2 * i + 1] += b; ydiag[2 * j] += g; ydiag[2 * j + 1] += b;
    auto& a = nb[i][j]; a.first -= g; a.second -= b;
    auto& c = nb[j][i]; c.first -= g; c.second -= b;
  }
  std::vector<int32_t> adj_ptr(n + 1, 0), adj_idx;
  std::vector<double> adj_y;
  for (int i = 0; i < n; ++i) {
    for (const auto& kv : nb[i]) { adj_idx.push_back(kv.first); adj_y.push_back(kv.second.first); adj_y.push_back(kv.second.second); }
    adj_ptr[i + 1] = (int32_t)adj_idx.size();
  }
  DeviceGuard guard(device);
  if (!guard.ok) return no_device();
  cudaDeviceProp prop;
  GFR_CUDA(cudaGetDeviceProperties(&prop, device));
  if ((N <= 127 ? dense_reg_smem_bytes(n, N) : dense_smem_bytes(n, N)) > (size_t)prop.sharedMemPerBlockOptin)
    return fail(GFR_E_LIMIT, "the dense Jacobian of this network exceeds the shared memory of an SM "
                             "(non-slack + PQ buses <= ~165); radial feeders take the tree-ordered solver");
  // pack: ints = bus_type | col_theta | col_vm | adj_ptr | adj_idx | line_from | line_to ; doubles (16-byte aligned
  // pairs first) = adj_y | ydiag | line_y | vm_set | line_rating
  std::vector<int32_t> ints;
  auto addi = [&](const int32_t* p, size_t c) { size_t o = ints.size(); ints.insert(ints.end(), p, p + c); return o; };
  const size_t o_bt = addi(d->bus_type, n), o_ct = addi(col_theta.data(), n), o_cv = addi(col_vm.data(), n),
               o_ap = addi(adj_ptr.data(), n + 1), o_ai = addi(adj_idx.data(), adj_idx.size()),
               o_lf = addi(d->line_from, m), o_lt = addi(d->line_to, m);
  std::vector<double> dbls;
  auto addd = [&](const double* p, size_t c) { size_t o = dbls.size(); dbls.insert(dbls.end(), p, p + c); return o; };
  const size_t o_ay = addd(adj_y.data(), adj_y.size()), o_yd = addd(ydiag.data(), ydiag.size()),
               o_ly = addd(line_y.data(), line_y.size()), o_vm = addd(d->vm_set, n), o_lr = addd(d->line_rating, m);
  auto* net = new gfr_network();
  net->device = device; net->sm_count = prop.multiProcessorCount; net->smem_optin = (int)prop.sharedMemPerBlockOptin;
  cudaError_t e1 = cudaMalloc(&net->d_ints, ints.size() * 4), e2 = cudaMalloc(&net->d_dbls, dbls.size() * 8);
  if (e1 == cudaSuccess) e1 = cudaMemcpy(net->d_ints, ints.data(), ints.size() * 4, cudaMemcpyHostToDevice);
  if (e2 == cudaSuccess) e2 = cudaMemcpy(net->d_dbls, dbls.data(), dbls.size() * 8, cudaMemcpyHostToDevice);
  if (e1 != cudaSuccess || e2 != cudaSuccess) { gfr_network_destroy(net); return cuda_fail(e1 != cudaSuccess ? e1 : e2, "cudaMalloc(network)"); }
  const int* di = (const int*)net->d_ints;
  const double* dd = (const double*)net->d_dbls;
  NetDev& nd = net->nd;
  nd.n = n; nd.m = m; nd.N = N; nd.n_theta = nt; nd.s_base = d->s_base;
  nd.bus_type = di + o_bt; nd.col_theta = di + o_ct; nd.col_vm = di + o_cv; nd.adj_ptr = di + o_ap;
  nd.adj_idx = di + o_ai; nd.line_from = di + o_lf; nd.line_to = di + o_lt;
  nd.adj_y = (const D2*)(dd + o_ay); nd.ydiag = (const D2*)(dd + o_yd); nd.line_y = (const D2*)(dd + o_ly);
  nd.vm_set = dd + o_vm; nd.line_rating = dd + o_lr;
  *out = net;
  return GFR_OK;
}

void gfr_network_destroy(gfr_network* net) {
  if (!net) return;
  DeviceGuard guard(net->device);
  cudaFree(net->d_ints);
  cudaFree(net->d_dbls);
  delete net;
}

int gfr_network_unknowns(const gfr_network* net) { return net ? net->nd.N : 0; }

int gfr_network_solve(const gfr_network* net, int64_t B, const double* p_inj, const gfr_solver_cfg* cfg,
                      const gfr_sol_out* out, void* stream) {
  return gfr_network_solve_pq(net, B, p_inj, nullptr, cfg, out, stream);
}

int gfr_network_solve_pq(const gfr_network* net, int64_t B, const double* p_inj, const double* q_inj,
                         const gfr_solver_cfg* cfg, const gfr_sol_out* out, void* stream) {
  if (!net || !p_inj || !cfg || !out) return fail(GFR_E_ARG, "null argument");
  if (B < 1) return fail(GFR_E_ARG, "B must be >= 1");
  if (int rc = check_stopping(cfg)) return rc;
  DeviceGuard guard(net->device);
  if (!guard.ok) return no_device();
  // kernel choice: [J | mismatch] in registers up to 127 unknowns (cfg->lanes: 0 = this choice, 1 = always the
  // shared-memory kernel, 2 = the register kernel or GFR_E_LIMIT); with q_inj, their specified-Q instantiations
  typedef void (*dense_fn)(const NetDev, const double, const int, const double, const double*, const SolOut, const long long);
  typedef void (*dense_pq_fn)(const NetDev, const double, const int, const double, const double*, const double*,
                              const SolOut, const long long);
  const int N = net->nd.N;
  if (cfg->lanes < 0 || cfg->lanes > 2) return fail(GFR_E_ARG, "lanes must be 0 (auto), 1 (shared-memory LU) or 2 (register LU) for a network solve");
  if (cfg->lanes == 2 && N > 127) return fail(GFR_E_LIMIT, "the register-resident elimination takes at most 127 unknowns");
  const bool in_regs = cfg->lanes != 1 && N <= 127;
  dense_fn fn = dense_solve_kernel;
  dense_pq_fn fn_pq = dense_solve_pq_kernel;
  int threads = N <= 48 ? 128 : 256;
  size_t smem = dense_smem_bytes(net->nd.n, N);
  if (in_regs) {
    smem = dense_reg_smem_bytes(net->nd.n, N);
    // 8 x TX threads, R = ceil(N / 8) register rows each: TX = 8 up to 56 unknowns, 16 up to 96, 32 above (measured
    // sweep, profiles/r01_tune_dense.txt).  R alone sets TX: 8 for R 1 - 7, 16 for R 8 - 12, 32 for R 13 - 16
#define K dense_solve_reg_kernel
    static const dense_fn by_r[] = { nullptr, K<8, 1>, K<8, 2>, K<8, 3>, K<8, 4>, K<8, 5>, K<8, 6>, K<8, 7>,
                                     K<16, 8>, K<16, 9>, K<16, 10>, K<16, 11>, K<16, 12>,
                                     K<32, 13>, K<32, 14>, K<32, 15>, K<32, 16> };
#undef K
#define K dense_solve_reg_pq_kernel
    static const dense_pq_fn by_r_pq[] = { nullptr, K<8, 1>, K<8, 2>, K<8, 3>, K<8, 4>, K<8, 5>, K<8, 6>, K<8, 7>,
                                           K<16, 8>, K<16, 9>, K<16, 10>, K<16, 11>, K<16, 12>,
                                           K<32, 13>, K<32, 14>, K<32, 15>, K<32, 16> };
#undef K
    const int tx = N <= 56 ? 8 : N <= 96 ? 16 : 32;
    fn = by_r[(N + 7) / 8];
    fn_pq = by_r_pq[(N + 7) / 8];
    threads = 8 * tx;
  }
  const void* kfn = q_inj ? (const void*)fn_pq : (const void*)fn;
  GFR_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, net->smem_optin));
  int per_sm = 0;
  GFR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kfn, threads, smem));
  if (per_sm < 1) return fail(GFR_E_LIMIT, "the dense Jacobian of this network exceeds the shared memory of an SM");
  long long grid = (long long)net->sm_count * per_sm;
  if (grid > B) grid = B;
  const EnvCfg k = env_cfg_of(cfg);
  if (q_inj) fn_pq<<<(int)grid, threads, smem, (cudaStream_t)stream>>>(net->nd, k.tol, k.max_it, k.accel, p_inj, q_inj, *out, (long long)B);
  else fn<<<(int)grid, threads, smem, (cudaStream_t)stream>>>(net->nd, k.tol, k.max_it, k.accel, p_inj, *out, (long long)B);
  g_launches.fetch_add(1);
  GFR_CUDA(cudaGetLastError());
  return GFR_OK;
}

int gfr_noise_fill(int device, int64_t B, int32_t n_slots, const uint64_t* seeds, const uint64_t* draws,
                   double* out, void* stream) {
  if (B < 1 || n_slots < 1 || !seeds || !draws || !out) return fail(GFR_E_ARG, "bad argument");
  DeviceGuard guard(device);
  if (!guard.ok) return no_device();
  long long total = B * (long long)n_slots;
  long long grid = (total + 255) / 256;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (grid > (long long)sms * 8) grid = (long long)sms * 8;
  noise_fill_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(B, n_slots, seeds, draws, out);
  g_launches.fetch_add(1);
  GFR_CUDA(cudaGetLastError());
  return GFR_OK;
}

int gfr_fp64_peak(int device, double* tflops) {
  if (!tflops) return fail(GFR_E_ARG, "null argument");
  DeviceGuard guard(device);
  if (!guard.ok) return no_device();
  cudaDeviceProp prop;
  GFR_CUDA(cudaGetDeviceProperties(&prop, device));
  const int threads = 256, blocks = prop.multiProcessorCount * 8, iters = 1 << 15;
  double* d_out = nullptr;
  GFR_CUDA(cudaMalloc((void**)&d_out, (size_t)blocks * threads * 8));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  double best_ms = 1e30;
  for (int rep = 0; rep < 5; ++rep) {             // the first repetitions warm the clocks up
    cudaEventRecord(e0, 0);
    dfma_peak_kernel<<<blocks, threads>>>(d_out, iters, 1.0 + rep);
    cudaEventRecord(e1, 0);
    cudaError_t es = cudaEventSynchronize(e1);
    g_launches.fetch_add(1);
    if (es != cudaSuccess) { cudaFree(d_out); return cuda_fail(es, "dfma_peak_kernel"); }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep >= 2 && ms < best_ms) best_ms = ms;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(d_out);
  *tflops = 2.0 * 8.0 * (double)iters * (double)blocks * threads / (best_ms * 1e-3) / 1e12;
  return GFR_OK;
}

}  // extern "C"
