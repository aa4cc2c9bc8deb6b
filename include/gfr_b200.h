/*
 * gfr_b200.h - C ABI of the B200-native batched GridEnvironment.step path.
 *
 * The reference (danieleschmidt/grid-fed-rl-gym) is pure Python and has no FFI; these
 * entry points are what a binding for its hot path would call.  Each one cites the
 * reference interface it replaces (paths relative to /root/reference/grid_fed_rl/).
 *
 * Conventions
 *   - every function returns 0 on success, a negative GFR_E_* code otherwise, never
 *     throws; gfr_last_error() gives the thread-local message of the last failure
 *   - all I/O buffers are CALLER-OWNED DEVICE pointers on the env's / feeder's device
 *     (e.g. torch.Tensor.data_ptr()); NULL output pointers are skipped.  The library owns
 *     only the compiled feeder and the persistent per-env state, released by *_destroy
 *   - calls are asynchronous on the given cudaStream_t (passed as void*); a handle is
 *     not thread-safe; there is no global mutable state
 *   - "ref order" = position in feeder.buses / feeder.lines of the (repaired) feeder;
 *     "level order" = position in the leaf -> root elimination schedule (what the kernels use)
 *   - there is NO CPU fallback: without a CUDA device every call fails with GFR_E_CUDA
 */
#ifndef GFR_B200_H
#define GFR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GFR_ABI_VERSION 1

enum {
  GFR_OK = 0,
  GFR_E_ARG = -1,      /* bad argument / inconsistent description */
  GFR_E_CUDA = -2,     /* CUDA runtime failure (message has the cudaError string) */
  GFR_E_LIMIT = -3     /* feeder too large for the compiled kernels' shared-memory plan */
};

enum { GFR_SOLVER_SWEEP = 0, GFR_SOLVER_NEWTON = 1 };
enum { GFR_BUS_SLACK = 0, GFR_BUS_PV = 1, GFR_BUS_PQ = 2 };
enum { GFR_GEN_SOLAR = 0, GFR_GEN_WIND = 1 };

typedef struct gfr_feeder gfr_feeder;   /* compiled topology, device resident */
typedef struct gfr_env gfr_env;         /* B environment instances on one device */

/* Host-side description of a radial feeder, arrays in LEVEL order: k = 0 is the ROOT of the
 * traversal tree (any bus; the tree's center halves the sequential depth of a feeder whose slack
 * bus sits at one end), every bus sits in a later level than its parent, levels may be capped to the number
 * of cooperating lanes.  The order only shapes the device-side traversal: results are always
 * reported in ref order.
 * Produced by grid_fed_rl_b200.topology.compile_feeder from feeder.buses / .lines / .loads /
 * .generators (reference feeders/base.py:30-52; Bus/Line/Load environments/base.py:197-295). */
typedef struct {
  int32_t n_bus, n_levels, n_load, n_gen, n_bat;
  int32_t n_pool;                   /* Newton: least number of shared-memory hand-off slots to provide (0 = as few as the
                                       library's own plan needs) */
  int32_t lanes_hint;               /* lanes the level schedule was capped for (levels hold at most this many buses);
                                       what `lanes = 0` resolves to.  0 = not said: gfr_auto_lanes decides */
  int32_t n_tie;                    /* loop-closing lines of a weakly meshed feeder (0: radial).  The feeder then has
                                       n - 1 + n_tie lines; sweep solver only */
  double s_base;                    /* VA; feeder.parameters.base_power * 1e6 */
  const int32_t* order;             /* [n]  level k -> ref bus index */
  const int32_t* parent;            /* [n]  level index of the parent, -1 for k = 0 */
  const int32_t* level_ptr;         /* [n_levels+1] */
  const int32_t* child_ptr;         /* [n+1] children of k are child_idx[child_ptr[k] .. child_ptr[k+1]) */
  const int32_t* child_idx;         /* [n-1] level indices of the children, parent by parent */
  const int32_t* lane_of;           /* [n]  Newton, optional: the lane (< lanes_hint) that eliminates bus k.  A bus
                                            eliminated right after one of its children on the same lane takes that
                                            child's contribution from registers.  NULL = position inside the level */
  const int32_t* bus_type;          /* [n]  GFR_BUS_* */
  const double* vm_set;             /* [n]  slack / pv voltage magnitude */
  const double* g;                  /* [n]  series conductance of branch (parent[k], k), k >= 1 */
  const double* b;                  /* [n]  series susceptance */
  const double* gdiag;              /* [n]  Re Y_kk (reference power_flow.py:48-73 accumulation order) */
  const double* bdiag;              /* [n]  Im Y_kk */
  const double* r;                  /* [n]  branch resistance, pu */
  const double* x;                  /* [n]  branch reactance, pu */
  const int32_t* line_of;           /* [n]  ref line index of branch k (-1 for k = 0); with tie_line a permutation of the lines */
  const int32_t* from_is_parent;    /* [n]  1 if line.from_bus is the parent end */
  const double* rating;             /* [n]  line rating, VA */
  const int32_t* load_bus;          /* [L]  level index */
  const double* load_base;          /* [L]  W  (Load.base_power) */
  const double* load_p;             /* [L]  W  static Load.active_power (obs, frequency model) */
  const double* load_q;             /* [L]  var static Load.reactive_power (obs) */
  const int32_t* gen_type;          /* [G]  GFR_GEN_* */
  const int32_t* gen_bus;           /* [G] */
  const double* gen_cap;            /* [G]  W */
  const double* gen_p0;             /* [G]  solar panel_area | wind cut_in_speed */
  const double* gen_p1;             /* [G]  solar efficiency | wind rated_speed */
  const double* gen_p2;             /* [G]  -                | wind cut_out_speed */
  const int32_t* bat_bus;           /* [Bt] */
  const double* bat_cap;            /* [Bt] BatteryModel.capacity */
  const double* bat_rating;         /* [Bt] BatteryModel.power_rating */
  const double* bat_eff;            /* [Bt] BatteryModel.efficiency */
  const double* bat_soc0;           /* [Bt] state of charge after reset (0.5) */
  const double* load_profile;       /* [24] TimeVaryingLoadModel.daily_profile (dynamics.py:43-48) */
  /* Ties: the lines that close a cycle (feeder.lines in list order, every line that joins two buses already
   * connected).  The traversal tree is the rest; the sweep restores the loops by compensation: one current per
   * tie (from -> to), corrected every iteration by tie_zinv x (V_from - V_to - z_tie J).  The reference takes
   * such networks through its dense Ybus (power_flow.py:48-73). */
  const int32_t* tie_line;          /* [t]  ref line index */
  const int32_t* tie_from;          /* [t]  level index of line.from_bus */
  const int32_t* tie_to;            /* [t]  level index of line.to_bus */
  const double* tie_r;              /* [t]  pu */
  const double* tie_x;              /* [t]  pu */
  const double* tie_rating;         /* [t]  VA */
  const double* tie_zinv;           /* [t, t, 2] inverse of the loop-impedance matrix, row-major (re, im):
                                            Z[i][j] = sum over tree branches on both loops of +-z + [i == j] z_tie */
} gfr_feeder_desc;

/* Solver settings: PowerFlowSolver.__init__(tolerance, max_iterations) + NewtonRaphsonSolver's
 * acceleration_factor (reference power_flow.py:28-35, :79-87). */
typedef struct {
  int32_t solver;                   /* GFR_SOLVER_* */
  int32_t max_iterations;
  double tolerance;                 /* newton: max |dP|,|dQ| (pu); sweep: max |dV| (pu) */
  double acceleration;              /* newton only; reference default 1.0 */
  int32_t lanes;                    /* 0 = auto; threads cooperating on one instance: 1..32 (part of a warp,
                                       feeder image staged in shared memory) or 64, 128, 256 (one CTA per
                                       instance, feeder image read from global memory) */
  int32_t reserved;
} gfr_solver_cfg;

/* GridEnvironment.__init__ kwargs (reference grid_env.py:161-174). */
typedef struct {
  double timestep;                  /* s */
  int32_t episode_length;
  int32_t stochastic_loads;         /* bool */
  int32_t weather_variation;        /* bool */
  int32_t reserved;
  double v_min, v_max;              /* voltage_limits */
  double f_min, f_max;              /* frequency_limits */
  double safety_penalty;
  double load_noise;                /* TimeVaryingLoadModel noise_factor, reference 0.1 */
  gfr_solver_cfg solver;
  int64_t env_id_offset;            /* global id of this env's instance 0 (a shard of a larger job): until a reset
                                       gives seeds, instance i draws from the Philox stream keyed env_id_offset + i */
} gfr_env_cfg;

/* Per-step results besides the observation (reference step() 5-tuple + info, grid_env.py:610-619). */
typedef struct {
  double* reward;                   /* [B] */
  uint8_t* terminated;              /* [B] */
  uint8_t* truncated;               /* [B] */
  uint8_t* error;                   /* [B] action rejected (NaN/Inf): reward = -2*safety_penalty, terminated */
  uint8_t* converged;               /* [B] info["power_flow_converged"] */
  int32_t* iterations;              /* [B] PowerFlowSolution.iterations */
  double* max_voltage;              /* [B] info["max_voltage"] */
  double* min_voltage;              /* [B] info["min_voltage"] */
  double* losses;                   /* [B] W, info["total_losses"] (= solution.losses) */
  double* max_mismatch;             /* [B] PowerFlowSolution.max_mismatch */
  uint8_t* violations;              /* [B,4] voltage_high, voltage_low, frequency_high, frequency_low */
  int32_t* violation_count;         /* [B] env.constraint_violations */
  int32_t* current_step;            /* [B] */
  double* episode_reward;           /* [B] */
  double* noise_used;               /* [B, 4+L] the noise row this step consumed (either mode) */
} gfr_step_out;

/* PowerFlowSolution fields (reference power_flow.py:12-22), batched, ref order. */
typedef struct {
  uint8_t* converged;               /* [B] */
  int32_t* iterations;              /* [B] */
  double* bus_voltages;             /* [B,n] */
  double* bus_angles;               /* [B,n] rad */
  double* line_flows;               /* [B,m] pu, from -> to */
  double* line_loadings;            /* [B,m] |S_ij| * s_base / rating */
  double* losses;                   /* [B] pu */
  double* max_mismatch;             /* [B] */
} gfr_sol_out;

int gfr_abi_version(void);
const char* gfr_last_error(void);

/* Compile a feeder description onto `device`.  Replaces the per-call Ybus build of
 * PowerFlowSolver.build_admittance_matrix (reference power_flow.py:48-73). */
int gfr_feeder_create(const gfr_feeder_desc* desc, int device, gfr_feeder** out);
void gfr_feeder_destroy(gfr_feeder* f);

/* GridEnvironment(feeder, **cfg) for n_envs instances (reference grid_env.py:161-241).
 * State after creation is the constructor's (wind 5, temperature 25, cloud 0.3, ...). */
int gfr_env_create(const gfr_feeder* f, int64_t n_envs, const gfr_env_cfg* cfg, gfr_env** out);
void gfr_env_destroy(gfr_env* e);
int64_t gfr_env_num_envs(const gfr_env* e);
int gfr_env_obs_dim(const gfr_env* e);      /* D = 2n + 2m + 1 + 2L + G + 2Bt (grid_env.py:307-314) */
int gfr_env_act_dim(const gfr_env* e);      /* A = Bt + G (grid_env.py:351) */
int gfr_env_noise_dim(const gfr_env* e);    /* 4 + L */
/* Library-owned observation buffer [B, D] fp64 row-major (get_observation, grid_env.py:753-783);
 * rewritten in place by reset and step (for an instance whose action was rejected only the
 * renewable outputs are refreshed; the rest of its state, hence of its observation, is unchanged). */
double* gfr_env_obs(gfr_env* e);
/* Make the env write its observations into a CALLER-OWNED device buffer [B, D] instead (the
 * current contents are copied over, the library's own buffer is released).  This is how a host
 * framework gets the observation as one of its own tensors without a copy per step. */
int gfr_env_bind_obs(gfr_env* e, double* obs, void* stream);
/* The same with a choice of type and, optionally, TWO alternating buffers: step t writes the buffer that does not
 * hold observation t - 1, so a caller can copy observation t - 1 out (to the host, to a replay block) on another
 * stream while step t runs.  dtype GFR_OBS_F32 makes the kernels write the observation as fp32 - the type the
 * reference declares for its observation space (grid_env.py:346) - halving what a host-side policy pulls over
 * PCIe; every other output stays fp64.  obs_b = NULL binds one buffer.  gfr_env_obs_current() is the buffer
 * holding the latest observation (reset writes into it, the next step into the other one). */
enum { GFR_OBS_F64 = 0, GFR_OBS_F32 = 1 };
int gfr_env_bind_obs_buffers(gfr_env* e, void* obs_a, void* obs_b, int dtype, void* stream);
void* gfr_env_obs_current(gfr_env* e);
/* Columns [col0, col0 + ncols) of every row of one of the bound observation buffers to a HOST buffer laid out
 * like the observation ([B, D], same item type; pinned memory for an asynchronous copy): one strided DMA on
 * `stream`.  A host-side policy uses it to leave the 2L static load columns (constants after construction,
 * grid_env.py:766-770) where they are and pull only what a step rewrote. */
int gfr_env_obs_to_host(gfr_env* e, const void* obs_device, void* host_dst, int32_t col0, int32_t ncols, void* stream);
/* How the step kernel is launched for this env (for benchmarks / profiles): threads cooperating
 * on one instance, threads per CTA, CTAs, dynamic shared memory per CTA. */
int gfr_env_launch_info(const gfr_env* e, int32_t* lanes, int32_t* threads, int32_t* grid,
                        int64_t* smem_bytes);
/* Size in bytes / copy of the persistent per-instance state (checkpoint / resume). */
int64_t gfr_env_state_bytes(const gfr_env* e);
int gfr_env_state_get(gfr_env* e, void* dst_device, void* stream);
int gfr_env_state_set(gfr_env* e, const void* src_device, void* stream);

/* GridEnvironment.reset(seed) (reference grid_env.py:360-408) for the instances with mask != 0
 * (mask NULL = all).  seeds [B] (NULL = keep each instance's stream) re-key the in-kernel
 * Philox stream.  noise [B,4] = the four weather draws reset consumes (NULL = Philox).
 * start_time = time of day (s) the first step starts from (the reference always uses 0). */
int gfr_env_reset(gfr_env* e, const uint64_t* seeds, const uint8_t* mask, const double* noise,
                  double start_time, void* stream);

/* The info of the instances a reset touched (reference grid_env.py:360-408: step and violation counters, episode
 * reward, losses back to zero, voltages at 1.0), written into the caller's output table `out` (the one gfr_env_step
 * fills; noise_used is left alone) for the instances with mask != 0 (mask NULL = all).  One launch. */
int gfr_env_reset_outputs(gfr_env* e, const uint8_t* mask, const gfr_step_out* out, void* stream);

/* GridEnvironment.step(action) (reference grid_env.py:410-619) for all B instances.
 * actions [B,A].  noise [B,4+L] (u_irradiance, z_wind, z_temperature, z_cloud, z_load_0..)
 * replays the reference's random.random / random.gauss / np.random.normal draws; NULL =
 * in-kernel Philox4x32-10 keyed (seed, draw counter, slot). */
int gfr_env_step(gfr_env* e, const double* actions, const double* noise, const gfr_step_out* out,
                 void* stream);

/* solver.solve(...) (reference power_flow.py:89-211) on B independent injection vectors.
 * p_inj [B,n] pu in ref bus order (generation minus load; the slack entry is ignored). */
int gfr_solve(const gfr_feeder* f, int64_t B, const double* p_inj, const gfr_solver_cfg* cfg,
              const gfr_sol_out* out, void* stream);
/* gfr_solve with specified reactive power: q_inj [B,n] pu in ref bus order (generation minus load, like p_inj).
 * The Q entries of the slack and of PV buses are ignored (those buses have no Q equation).  q_inj = NULL is
 * gfr_solve: Q_spec = 0 through the same kernels.  p_inj = NULL -> GFR_E_ARG. */
int gfr_solve_pq(const gfr_feeder* f, int64_t B, const double* p_inj, const double* q_inj,
                 const gfr_solver_cfg* cfg, const gfr_sol_out* out, void* stream);

/* ---- meshed networks: the reference's dense Newton-Raphson as written ------------------------
 * NewtonRaphsonSolver.solve on ANY connected network (cycles allowed): dense Ybus
 * (power_flow.py:48-73, an impedance of magnitude <= 1e-12 is an open line), dense polar Jacobian
 * (power_flow.py:213-295, deviation D2), LU with partial pivoting = np.linalg.solve / LAPACK dgesv
 * (power_flow.py:187), one CTA per instance with the Jacobian in shared memory.  Bus and line order
 * are the caller's (no renumbering).  Limit: (#non-slack + #PQ buses) <= ~165, else GFR_E_LIMIT -
 * radial feeders of any size take gfr_solve. */
typedef struct gfr_network gfr_network;
typedef struct {
  int32_t n_bus, n_line;
  double s_base;                    /* VA: line_loadings = |S| s_base / rating (deviation D1) */
  const int32_t* bus_type;          /* [n_bus] GFR_BUS_* (exactly one slack) */
  const double* vm_set;             /* [n_bus] bus.voltage_magnitude (used for slack / PV buses) */
  const int32_t* line_from;         /* [n_line] index into the buses */
  const int32_t* line_to;           /* [n_line] */
  const double* line_r;             /* [n_line] pu */
  const double* line_x;             /* [n_line] pu */
  const double* line_rating;        /* [n_line] VA */
} gfr_network_desc;
int gfr_network_create(const gfr_network_desc* desc, int device, gfr_network** out);
void gfr_network_destroy(gfr_network* net);
int gfr_network_unknowns(const gfr_network* net);          /* order of the dense Jacobian */
/* p_inj [B, n_bus] pu (generation minus load, Q_spec = 0 as the reference); out arrays in the
 * caller's bus / line order; cfg->solver is ignored; cfg->lanes picks the kernel: 0 = automatic ([J | mismatch]
 * held in registers up to 127 unknowns, in shared memory above), 1 = always shared memory, 2 = registers or
 * GFR_E_LIMIT. */
int gfr_network_solve(const gfr_network* net, int64_t B, const double* p_inj, const gfr_solver_cfg* cfg,
                      const gfr_sol_out* out, void* stream);
/* gfr_network_solve with specified reactive power q_inj [B, n_bus] pu (NULL: Q_spec = 0, as gfr_network_solve);
 * the slack's and PV buses' entries are ignored. */
int gfr_network_solve_pq(const gfr_network* net, int64_t B, const double* p_inj, const double* q_inj,
                         const gfr_solver_cfg* cfg, const gfr_sol_out* out, void* stream);

/* The noise rows the in-kernel generator yields: out [B, n_slots] for keys seeds[B] and draw
 * counters draws[B] (slot 0 uniform, slots 1.. standard normal). */
int gfr_noise_fill(int device, int64_t B, int32_t n_slots, const uint64_t* seeds,
                   const uint64_t* draws, double* out, void* stream);

/* Measured FP64 FMA throughput of the device (TFLOP/s, 2 flop per DFMA): the denominator for the
 * FP64 side of the roofline, which the driver-written MEASURED_PEAKS.json does not carry. */
int gfr_fp64_peak(int device, double* tflops);

/* Threads cooperating on one instance when `lanes = 0` and the description carries no lanes_hint: the measured
 * rule (n_bus, GFR_SOLVER_*, depth = levels of the tree rooted at its center, 0 if unknown).  The one copy of it:
 * grid_fed_rl_b200.topology.auto_lanes calls this. */
int gfr_auto_lanes(int n_bus, int solver, int depth);

/* Launch bookkeeping for benchmarks: kernels launched by this library since load. */
int64_t gfr_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* GFR_B200_H */
