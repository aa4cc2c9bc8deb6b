// gfr_dense.cuh - Newton-Raphson load flow on an ARBITRARY (meshed) network: one CTA per
// instance, the dense polar Jacobian assembled in shared memory and factorised there by Gaussian
// elimination with partial pivoting.  This is the reference's algorithm as written - dense
// (2(n-1))^2 system, np.linalg.solve = LAPACK dgesv - for the networks the tree-ordered kernels of
// gfr_device.cuh cannot take (cycles: SyntheticFeeder(connectivity > 0), the shipped IEEE feeders
// with their loop-closing lines kept).  Size limit: the Jacobian has to fit the shared memory of an
// SM, N = (#non-slack) + (#PQ) <= ~165.
//
// Reference (paths under /root/reference/grid_fed_rl/):
//   Ybus                  environments/power_flow.py:48-73   (|z| <= 1e-12 -> open line)
//   Newton-Raphson        environments/power_flow.py:89-211  (flat start; check, then update)
//   Jacobian              environments/power_flow.py:213-295 (+ deviation D2, DESIGN.md); unknowns
//                         ordered as there: angles of the non-slack buses, then |V| of the PQ buses
//   solve                 environments/power_flow.py:187     (np.linalg.solve -> dgesv: LU, partial pivoting)
//   update                environments/power_flow.py:297-327
//   line flows / losses   environments/power_flow.py:329-358, :199-200
#pragma once
#include "gfr_device.cuh"

namespace gfr {

// Device-resident network (bus / line order = the caller's, no renumbering)
struct NetDev {
  int n, m, N, n_theta;           // buses, lines, unknowns, angle unknowns (= non-slack buses)
  double s_base;
  const int* bus_type;            // [n]
  const int* col_theta;           // [n] column (= row) of the bus's angle unknown, -1 for the slack
  const int* col_vm;              // [n] column (= row) of the bus's |V| unknown, -1 unless PQ
  const int* adj_ptr;             // [n + 1] neighbours of a bus, parallel lines merged
  const int* adj_idx;             // [nnz]
  const D2* adj_y;                // [nnz] (G_ij, B_ij) = -(sum of the series admittances between i and j)
  const D2* ydiag;                // [n]   (G_ii, B_ii)
  const double* vm_set;           // [n]
  const int* line_from;           // [m]
  const int* line_to;             // [m]
  const D2* line_y;               // [m] series g + jb (0 for an open line)
  const double* line_rating;      // [m]
};

GFR_HD size_t dense_smem_bytes(int n, int N) {
  const size_t ld = (size_t)(N | 1);                        // odd leading dimension: conflict-free column walks
  return ld * (size_t)N * 8 + (size_t)N * 8 + (size_t)n * 32 + 64 * 8;
}

#if defined(__CUDACC__)

// NaN-propagating maximum over the CTA (numpy's max); every thread gets the result
__device__ __forceinline__ double block_max_nan(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double w = __shfl_xor_sync(0xffffffffu, v, o);
    v = (w > v || w != w) ? w : v;
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  v = red[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { const double x = red[w]; v = (x > v || x != x) ? x : v; }
  return v;
}

// ---- the pieces both kernels share ------------------------------------------------------------------------

// flat start (:103, :131): 1.0 at 0 rad, slack / PV buses at their set magnitude
__device__ __forceinline__ void dense_flat_start(const NetDev& net, D2* ef, int tid, int nt) {
  for (int i = tid; i < net.n; i += nt) {
    D2 v;
    v.x = net.bus_type[i] == BUS_PQ ? 1.0 : net.vm_set[i];
    v.y = 0.0;
    ef[i] = v;
  }
}

// calculated injections and mismatch (:150-166); returns the NaN-propagating maximum over the CTA.
// SPEC_Q: PQ buses have a specified Q (qspec); without it Q_spec = 0, as in the reference.
template <bool SPEC_Q = false>
__device__ __forceinline__ double dense_mismatch(const NetDev& net, const D2* ef, D2* pq, double* rhs,
                                                 const double* __restrict__ pspec, const double* __restrict__ qspec,
                                                 double* red, int tid, int nt) {
  double mm = 0.0;
  for (int i = tid; i < net.n; i += nt) {
    const D2 vi = ef[i];
    const D2 yd = net.ydiag[i];
    const double v2 = fma(vi.x, vi.x, vi.y * vi.y);
    double P = yd.x * v2, Q = -yd.y * v2;
    for (int q = net.adj_ptr[i]; q < net.adj_ptr[i + 1]; ++q) {
      const D2 vj = ef[net.adj_idx[q]];
      const D2 y = net.adj_y[q];
      const double a = fma(vi.x, vj.x, vi.y * vj.y), s = fma(vi.y, vj.x, -vi.x * vj.y);
      P = fma(y.x, a, fma(y.y, s, P));
      Q = fma(y.x, s, fma(-y.y, a, Q));
    }
    D2 c; c.x = P; c.y = Q;
    pq[i] = c;
    const int rt = net.col_theta[i], rv = net.col_vm[i];
    double aP = 0.0, aQ = 0.0;
    if (rt >= 0) { const double d = pspec[i] - P; rhs[rt] = d; aP = fabs(d); }
    if (rv >= 0) { const double d = (SPEC_Q ? qspec[i] : 0.0) - Q; rhs[rv] = d; aQ = fabs(d); }
    const double loc = (aQ > aP || aQ != aQ) ? aQ : aP;
    mm = (loc > mm || loc != loc) ? loc : mm;
  }
  return block_max_nan(mm, red);
}

// Jacobian (:213-295 with D2) into shared memory, column-major; |V| columns scaled by |V| (the polar
// update undoes it).  Ends with a CTA barrier.
__device__ __forceinline__ void dense_jacobian(const NetDev& net, const D2* ef, const D2* pq, double* J, int ld,
                                               int tid, int nt) {
  const int N = net.N;
  for (int q = tid; q < ld * N; q += nt) J[q] = 0.0;
  __syncthreads();
  for (int i = tid; i < net.n; i += nt) {
    const int rt = net.col_theta[i], rv = net.col_vm[i];
    if (rt < 0) continue;
    const D2 vi = ef[i];
    const D2 yd = net.ydiag[i];
    const D2 c = pq[i];
    const double v2 = fma(vi.x, vi.x, vi.y * vi.y);
    J[rt + rt * ld] = fma(-yd.y, v2, -c.y);                        // dP/dtheta:    -Q - B v2
    if (rv >= 0) {
      J[rt + rv * ld] = fma(yd.x, v2, c.x);                        // V dP/dV:       P + G v2
      J[rv + rt * ld] = fma(-yd.x, v2, c.x);                       // dQ/dtheta:     P - G v2
      J[rv + rv * ld] = fma(-yd.y, v2, c.y);                       // V dQ/dV:       Q - B v2
    }
    for (int q = net.adj_ptr[i]; q < net.adj_ptr[i + 1]; ++q) {
      const int j = net.adj_idx[q];
      const int ct = net.col_theta[j], cv = net.col_vm[j];
      if (ct < 0) continue;                                          // the slack has no unknowns
      const D2 vj = ef[j];
      const D2 y = net.adj_y[q];
      const double a = fma(vi.x, vj.x, vi.y * vj.y), s = fma(vi.y, vj.x, -vi.x * vj.y);
      const double al = fma(y.x, s, -y.y * a);                       // |Vi||Vj| (G sin - B cos)
      const double ga = fma(y.x, a, y.y * s);                        // |Vi||Vj| (G cos + B sin)
      J[rt + ct * ld] = al;
      if (cv >= 0) J[rt + cv * ld] = ga;
      if (rv >= 0) {
        J[rv + ct * ld] = -ga;
        if (cv >= 0) J[rv + cv * ld] = al;
      }
    }
  }
  __syncthreads();
}

// Mismatch and Jacobian in ONE pass over the adjacency lists (the register kernel): the same arithmetic, term
// by term, as dense_mismatch + dense_jacobian; J must be zero on entry (the caller clears it while the
// elimination result is scattered).  The Jacobian of the converged iterate is wasted, once per solve.
template <bool SPEC_Q = false>
__device__ __forceinline__ double dense_mismatch_jacobian(const NetDev& net, const D2* ef, double* J, int ld,
                                                          double* rhs, const double* __restrict__ pspec,
                                                          const double* __restrict__ qspec,
                                                          double* red, int tid, int nt) {
  double mm = 0.0;
  for (int i = tid; i < net.n; i += nt) {
    const D2 vi = ef[i];
    const D2 yd = net.ydiag[i];
    const int rt = net.col_theta[i], rv = net.col_vm[i];
    const double v2 = fma(vi.x, vi.x, vi.y * vi.y);
    double P = yd.x * v2, Q = -yd.y * v2;
    for (int q = net.adj_ptr[i]; q < net.adj_ptr[i + 1]; ++q) {
      const int j = net.adj_idx[q];
      const D2 vj = ef[j];
      const D2 y = net.adj_y[q];
      const double a = fma(vi.x, vj.x, vi.y * vj.y), s = fma(vi.y, vj.x, -vi.x * vj.y);
      P = fma(y.x, a, fma(y.y, s, P));
      Q = fma(y.x, s, fma(-y.y, a, Q));
      const int ct = net.col_theta[j], cv = net.col_vm[j];
      if (rt < 0 || ct < 0) continue;                                  // the slack has no equations / unknowns
      const double al = fma(y.x, s, -y.y * a);                         // |Vi||Vj| (G sin - B cos)
      const double ga = fma(y.x, a, y.y * s);                          // |Vi||Vj| (G cos + B sin)
      J[rt + ct * ld] = al;
      if (cv >= 0) J[rt + cv * ld] = ga;
      if (rv >= 0) {
        J[rv + ct * ld] = -ga;
        if (cv >= 0) J[rv + cv * ld] = al;
      }
    }
    double aP = 0.0, aQ = 0.0;
    if (rt >= 0) {
      const double d = pspec[i] - P;
      rhs[rt] = d; aP = fabs(d);
      J[rt + rt * ld] = fma(-yd.y, v2, -Q);                          // dP/dtheta:    -Q - B v2
      if (rv >= 0) {
        J[rt + rv * ld] = fma(yd.x, v2, P);                          // V dP/dV:       P + G v2
        J[rv + rt * ld] = fma(-yd.x, v2, P);                         // dQ/dtheta:     P - G v2
        J[rv + rv * ld] = fma(-yd.y, v2, Q);                         // V dQ/dV:       Q - B v2
      }
    }
    if (rv >= 0) { const double d = (SPEC_Q ? qspec[i] : 0.0) - Q; rhs[rv] = d; aQ = fabs(d); }
    const double loc = (aQ > aP || aQ != aQ) ? aQ : aP;
    mm = (loc > mm || loc != loc) ? loc : mm;
  }
  return block_max_nan(mm, red);
}

// polar update (:297-327): theta += a dtheta, |V| += a d|V|  <=>  V *= (1 + a x_v) e^{j a x_theta}.  Ends with a barrier.
__device__ __forceinline__ void dense_polar_update(const NetDev& net, D2* ef, const double* x, double accel,
                                                   int tid, int nt) {
  for (int i = tid; i < net.n; i += nt) {
    const int ct = net.col_theta[i], cv = net.col_vm[i];
    if (ct < 0) continue;
    double sn, cs;
    sincos_small(accel * x[ct], &sn, &cs);
    const double sc = cv >= 0 ? fma(accel, x[cv], 1.0) : 1.0;
    const D2 v = ef[i];
    D2 w;
    w.x = sc * fma(v.x, cs, -v.y * sn);
    w.y = sc * fma(v.x, sn, v.y * cs);
    ef[i] = w;
  }
  __syncthreads();
}

// results in the caller's bus / line order.  Ends with a barrier.
__device__ __forceinline__ void dense_results(const NetDev& net, const D2* ef, double* red, const SolOut& o,
                                              long long env, int converged, int iterations, double max_mismatch,
                                              int tid, int nt) {
  const int n = net.n, m = net.m;
  for (int i = tid; i < n; i += nt) {
    const D2 v = ef[i];
    if (o.bus_voltages) o.bus_voltages[env * n + i] = sqrt(v.x * v.x + v.y * v.y);
    if (o.bus_angles) o.bus_angles[env * n + i] = atan2_bus(v.y, v.x);
  }
  double loss = 0.0;
  for (int li = tid; li < m; li += nt) {
    const D2 vf = ef[net.line_from[li]], vt = ef[net.line_to[li]];
    const D2 y = net.line_y[li];
    const double de = vf.x - vt.x, df = vf.y - vt.y;
    const double ir = y.x * de - y.y * df, ii = y.x * df + y.y * de;      // I = y (V_from - V_to)
    const double P = vf.x * ir + vf.y * ii, Q = vf.y * ir - vf.x * ii;    // V_from conj(I)
    loss += y.x * (de * de + df * df);                                    // Re sum_i V_i conj((YV)_i), line by line
    const double rating = net.line_rating[li];
    if (o.line_flows) o.line_flows[env * m + li] = P;
    if (o.line_loadings) o.line_loadings[env * m + li] = rating > 0.0 ? sqrt(P * P + Q * Q) * net.s_base / rating : 0.0;
  }
  {   // deterministic sum over the CTA
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, off);
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = loss;
    __syncthreads();
    loss = 0.0;
    for (int w = 0; w < ((nt + 31) >> 5); ++w) loss += red[w];
  }
  if (tid == 0) {
    if (o.losses) o.losses[env] = loss;
    if (o.max_mismatch) o.max_mismatch[env] = max_mismatch;
    if (o.converged) o.converged[env] = (uint8_t)converged;
    if (o.iterations) o.iterations[env] = iterations;
  }
  __syncthreads();
}

// "better pivot" order shared by the searches: a NaN wins and sticks (numpy / idamax on NaN input), then the
// larger magnitude, then the lower row index
__device__ __forceinline__ bool pivot_takes(double ob, int oi, double best, int bi) {
  return (ob != ob && !(best != best)) || (!(best != best) && (ob > best || (ob == best && oi < bi)));
}

// ---- kernel 1: Jacobian factorised in shared memory (any N that fits; used for N >= 128) ---------------------
// (SPEC_Q: q_inj [B, n] specified Q at the PQ buses; dense_solve_pq_kernel)
template <bool SPEC_Q>
__device__ __forceinline__ void dense_solve(const NetDev& net, const double tol, const int max_it, const double accel,
                                            const double* __restrict__ p_inj, const double* __restrict__ q_inj,
                                            const SolOut& o, const long long B) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int n = net.n, N = net.N;
  const int ld = N | 1;
  double* J = reinterpret_cast<double*>(smem);               // column-major, J[r + c * ld]
  double* rhs = J + (size_t)ld * N;                          // [N] mismatch, then the corrections
  D2* ef = reinterpret_cast<D2*>(rhs + N);                   // [n] e + jf   (16-byte aligned: ld is odd, so (ld + 1) N doubles is even)
  D2* pq = ef + n;                                           // [n] calculated (P, Q)
  double* red = reinterpret_cast<double*>(pq + n);           // [64] reductions, pivot search
  int* redi = reinterpret_cast<int*>(red + 32);
  const int tid = threadIdx.x, nt = blockDim.x;

  for (long long env = blockIdx.x; env < B; env += gridDim.x) {
    const double* pspec = p_inj + env * n;
    const double* qspec = SPEC_Q ? q_inj + env * n : nullptr;
    dense_flat_start(net, ef, tid, nt);
    __syncthreads();
    int converged = 0, iterations = max_it;
    double max_mismatch = INFINITY;
    for (int it = 0; it < max_it; ++it) {
      const double mm = dense_mismatch<SPEC_Q>(net, ef, pq, rhs, pspec, qspec, red, tid, nt);
      max_mismatch = mm;
      if (mm < tol) { converged = 1; iterations = it + 1; break; }      // checked before the update (:168-171)
      dense_jacobian(net, ef, pq, J, ld, tid, nt);
      // ---- Gaussian elimination with partial pivoting on [J | rhs] (dgesv, :187).  Two CTA barriers per
      //      pivot column: the multipliers are formed on the fly (nothing reuses L: the right-hand side is
      //      eliminated in the same sweep), and the warp that updates column k + 1 finds that column's
      //      pivot - largest |entry|, the first among equals (idamax) - before the barrier that ends step k.
      int singular = 0;
      {
        // pivot of column 0 by warp 0
        if (tid < 32) {
          double best = -1.0;
          int bi = 0;
          for (int i = tid; i < N; i += 32) {
            const double a = fabs(J[i]);
            if ((a > best || a != a) && !(best != best)) { best = a; bi = i; }
          }
#pragma unroll
          for (int off = 16; off > 0; off >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, off);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
            if (pivot_takes(ob, oi, best, bi)) { best = ob; bi = oi; }
          }
          if (tid == 0) { red[0] = best; redi[0] = bi; }
        }
        __syncthreads();
      }
      for (int k = 0; k < N; ++k) {
        const double best = red[0];
        const int bi = redi[0];
        if (!(best > 0.0) && !(best != best)) { singular = 1; break; }   // exact-zero pivot (:188-190); NaN runs on
        __syncthreads();                                                 // red is rewritten at the end of this step
        if (bi != k) {
          for (int c = k + tid; c <= N; c += nt) {
            double* pa = c < N ? &J[k + c * ld] : &rhs[k];
            double* pb = c < N ? &J[bi + c * ld] : &rhs[bi];
            const double t = *pa; *pa = *pb; *pb = t;
          }
          __syncthreads();
        }
        const double rp = 1.0 / J[k + k * ld];
        {
          const int tx = tid & 31, ty = tid >> 5, ny = nt >> 5;
          for (int c = k + 1 + ty; c <= N; c += ny) {
            double* col = c < N ? &J[c * ld] : rhs;
            const double u = col[k];
            double nbest = -1.0;
            int nbi = k + 1;
            for (int i = k + 1 + tx; i < N; i += 32) {
              const double v = fma(-(J[i + k * ld] * rp), u, col[i]);    // multiplier = entry x (1 / pivot), as dgetf2
              col[i] = v;
              const double a = fabs(v);
              if ((a > nbest || a != a) && !(nbest != nbest)) { nbest = a; nbi = i; }
            }
            if (c == k + 1 && c < N) {                                   // warp 0, first column of its sweep: the next pivot
#pragma unroll
              for (int off = 16; off > 0; off >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, nbest, off);
                const int oi = __shfl_xor_sync(0xffffffffu, nbi, off);
                if (pivot_takes(ob, oi, nbest, nbi)) { nbest = ob; nbi = oi; }
              }
              if (tx == 0) { red[0] = nbest; redi[0] = nbi; }
            }
          }
        }
        __syncthreads();
      }
      if (singular) { iterations = it + 1; break; }
      // ---- back substitution by warp 0 alone (warp barriers instead of 2 N CTA barriers):
      //      x_k = rhs_k / U_kk, then rhs_i -= U_ik x_k above it
      if (tid < 32) {
        for (int k = N - 1; k >= 0; --k) {
          const double xk = rhs[k] / J[k + k * ld];
          __syncwarp();
          if (tid == 0) rhs[k] = xk;
          for (int i = tid; i < k; i += 32) rhs[i] = fma(-J[i + k * ld], xk, rhs[i]);
          __syncwarp();
        }
      }
      __syncthreads();
      dense_polar_update(net, ef, rhs, accel, tid, nt);
    }
    dense_results(net, ef, red, o, env, converged, iterations, max_mismatch, tid, nt);
  }
}
__global__ void __launch_bounds__(256)
dense_solve_kernel(const NetDev net, const double tol, const int max_it, const double accel,
                   const double* __restrict__ p_inj, const SolOut o, const long long B) {
  dense_solve<false>(net, tol, max_it, accel, p_inj, nullptr, o, B);
}
__global__ void __launch_bounds__(256)
dense_solve_pq_kernel(const NetDev net, const double tol, const int max_it, const double accel,
                      const double* __restrict__ p_inj, const double* __restrict__ q_inj, const SolOut o,
                      const long long B) {
  dense_solve<true>(net, tol, max_it, accel, p_inj, q_inj, o, B);
}

// ---- kernel 2: [J | mismatch] in REGISTERS, N <= 127 ----------------------------------------------------------
// The CTA is an 8 x TX grid of threads (thread = tx * 8 + ty, so the 8 threads that share a column are
// neighbouring lanes of one warp); thread (ty, tx) owns the entries (8 r + ty, c TX + tx) of the N x (N + 1)
// system, R x C of them, in registers (R = ceil(N / 8): one instantiation per R and TX).  Gauss-Jordan
// elimination with partial pivoting: the column is cleared in EVERY other row, so there is no back substitution
// and no L or U to keep - after N steps row p_k holds x_k x pivot_k in the right-hand-side column.  Rows are
// never swapped (a bit mask remembers the used ones).  The elimination is a chain of N dependent steps, so what
// counts is the latency of one step; it has ONE CTA barrier:
//   * the 8 owners of column k publish it (double-buffered) and look for its pivot with one redux.sync on a
//     32-bit key = the upper word of |x| with its low 7 bits replaced by 127 - row: the largest magnitude to 13
//     mantissa bits, the lowest row among equals, a NaN beats everything (as numpy's / idamax's NaN handling).
//     That is threshold pivoting with threshold 1 - 2^-13: any such row is as good a pivot as dgetf2's.  The
//     winning lane zeroes its own entry of the published column (so the pivot row is "cleared" by a multiplier
//     of zero), and publishes the row and the pivot; a column of zeros (all upper words < 128: zeros and the
//     deepest subnormals) is the reference's singular-matrix break (:188-190);
//   * barrier;
//   * the pivot row reaches the threads of its column group by warp shuffle (same tx = same warp; the row's
//     register is picked by a CTA-uniform switch) and is scaled by -1 / pivot once;
//   * every thread clears its R x C tile: one shared-memory load and up to C FMAs per row.  The local column
//     index is static: after TX steps block column kb is dead and the tile shifts left by one, so column k is
//     always local column 0; dead and padding columns are skipped by a CTA-uniform switch on the number of live
//     local columns.
GFR_HD size_t dense_reg_smem_bytes(int n, int N) {
  return dense_smem_bytes(n, N) + (size_t)(3 * 128) * 8 + (size_t)128 * 4 + 64;
}

#define GFR_ROW_CASE(i) case i: if constexpr (R > i) { _Pragma("unroll") for (int c = 0; c < C; ++c) un[c] = __shfl_sync(0xffffffffu, a[i < R ? i : 0][c], src); } break;

// Shared-memory mailboxes of the elimination
struct GJBoxes {
  double* Lbuf;      // [2][128] published pivot columns
  double* pvv;       // [2] pivot
  int* pvi;          // [2] pivot row, -1 = singular
  double* piv;       // [128] pivot of the step that used the row
  int* kof;          // [128] the step that used the row
};

// The pivot steps of one block column (columns k0 .. k0 + steps - 1 = local column 0 of thread columns
// 0 .. steps - 1) with CC live local columns.  Returns false on a singular matrix.
template <int TX, int R, int C, int CC>
__device__ __forceinline__ bool gj_block(double (&a)[R][C], unsigned& used, const GJBoxes& bx, const int k0,
                                         const int steps, const int ty, const int tx, const unsigned gmask,
                                         const int lane_base) {
  for (int kt = 0; kt < steps; ++kt) {
    const int k = k0 + kt;
    double* Lb = bx.Lbuf + (k & 1) * 128 + ty;
    if (tx == kt) {                                      // the 8 owners of column k (local column 0)
      unsigned bk = 0u;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        Lb[r * 8] = a[r][0];
        const unsigned h = ((unsigned)__double2hiint(a[r][0]) & 0x7fffff80u) | (unsigned)(127 - r * 8 - ty);
        bk = max(bk, ((used >> r) & 1u) ? 0u : h);
      }
      const unsigned mk = __reduce_max_sync(gmask, bk);
      if (mk < 128u) {
        if (ty == 0) bx.pvi[k & 1] = -1;
      } else if (bk == mk) {
        const int p = 127 - (int)(mk & 127u);
        double* mine = bx.Lbuf + (k & 1) * 128 + p;
        const double piv = *mine;
        *mine = 0.0;
        bx.pvv[k & 1] = piv;
        bx.pvi[k & 1] = p;
        bx.kof[p] = k;
        bx.piv[p] = piv;
      }
    }
    __syncthreads();
    const int p = bx.pvi[k & 1];
    const double piv = bx.pvv[k & 1];
    if (p < 0) return false;                             // CTA-uniform
    const double ap = fabs(piv);                         // the reciprocal overlaps the row broadcast below
    const double rp = (ap > 1e-280 && ap < 1e280) ? rcp_fast(piv) : 1.0 / piv;
    const int pr = p >> 3, pty = p & 7;
    if (ty == pty) used |= 1u << pr;
    // the pivot row, for this thread's columns: from lane pty of the column group
    double un[C];
    const int src = lane_base + pty;
    switch (pr) {
      GFR_ROW_CASE(0) GFR_ROW_CASE(1) GFR_ROW_CASE(2) GFR_ROW_CASE(3) GFR_ROW_CASE(4) GFR_ROW_CASE(5)
      GFR_ROW_CASE(6) GFR_ROW_CASE(7) GFR_ROW_CASE(8) GFR_ROW_CASE(9) GFR_ROW_CASE(10) GFR_ROW_CASE(11)
      GFR_ROW_CASE(12) GFR_ROW_CASE(13) GFR_ROW_CASE(14) GFR_ROW_CASE(15)
      default: break;
    }
#pragma unroll
    for (int c = 0; c < CC; ++c) un[c] *= -rp;
    if (tx <= kt) un[0] = 0.0;                           // local column 0 at or left of the pivot column: dead
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const double l = Lb[r * 8];
#pragma unroll
      for (int c = 0; c < CC; ++c) a[r][c] = fma(l, un[c], a[r][c]);
    }
  }
  return true;
}
#undef GFR_ROW_CASE

#define GFR_LIVE_CASE(i) case i: if constexpr (C >= i) ok = gj_block<TX, R, C, (C >= i ? i : 1)>(a, used, bx, k0, steps, ty, tx, gmask, lane_base); break;

// CTAs per SM the register kernel is compiled for.  Small tiles: the tile plus ~56 registers of everything
// else (measured: +5 % at 16 - 26 unknowns); larger ones are left to ptxas (a cap made them spill: -12 % at 38)
constexpr int dense_reg_min_blocks(int TX, int R) {
  const int C = 8 * R / TX + 1, regs = (2 * R * C + 56 + 7) / 8 * 8, b = 65536 / (8 * TX * regs);
  return regs > 96 ? 0 : b > 24 ? 24 : b;   // 0 = no request
}

template <int TX, int R, bool SPEC_Q>
__device__ __forceinline__ void dense_solve_reg(const NetDev& net, const double tol, const int max_it,
                                                const double accel, const double* __restrict__ p_inj,
                                                const double* __restrict__ q_inj, const SolOut& o, const long long B) {
  constexpr int TY = 8, C = 8 * R / TX + 1, nt = TY * TX;
  static_assert(R >= 1 && R <= 16 && C >= 1 && C <= 10 && nt % 32 == 0, "8 R rows <= 128; whole warps");
  extern __shared__ __align__(16) unsigned char smem[];
  const int n = net.n, N = net.N;
  const int ld = N | 1;
  double* J = reinterpret_cast<double*>(smem);               // assembly area, column-major; column N = rhs
  double* rhs = J + (size_t)ld * N;
  D2* ef = reinterpret_cast<D2*>(rhs + N);
  D2* pq = ef + n;
  double* red = reinterpret_cast<double*>(pq + n);           // [64]: 0..31 reductions, 32.. pivot mailbox
  GJBoxes bx;
  bx.pvv = red + 32;
  bx.pvi = reinterpret_cast<int*>(red + 34);
  bx.Lbuf = red + 64;
  bx.piv = bx.Lbuf + 256;
  bx.kof = reinterpret_cast<int*>(bx.piv + 128);
  const int tid = threadIdx.x;
  const int ty = tid % TY, tx = tid / TY;
  const unsigned gmask = 0xffu << ((tid & 31) & ~7);
  const int lane_base = (tid & 31) & ~7;

  for (long long env = blockIdx.x; env < B; env += gridDim.x) {
    const double* pspec = p_inj + env * n;
    const double* qspec = SPEC_Q ? q_inj + env * n : nullptr;
    dense_flat_start(net, ef, tid, nt);
    for (int q = tid; q < ld * N; q += nt) J[q] = 0.0;
    __syncthreads();
    int converged = 0, iterations = max_it;
    double max_mismatch = INFINITY;
    for (int it = 0; it < max_it; ++it) {
      const double mm = dense_mismatch_jacobian<SPEC_Q>(net, ef, J, ld, rhs, pspec, qspec, red, tid, nt);   // ends with a barrier
      max_mismatch = mm;
      if (mm < tol) { converged = 1; iterations = it + 1; break; }
      double a[R][C];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
          const int row = r * TY + ty, col = c * TX + tx;
          a[r][c] = (row < N && col <= N) ? J[row + col * ld] : 0.0;
        }
      unsigned used = 0;                                     // rows that may not become a pivot (used, or beyond N)
#pragma unroll
      for (int r = 0; r < R; ++r) if (r * TY + ty >= N) used |= 1u << r;
      bool ok = true;
      for (int kb = 0; kb * TX < N && ok; ++kb) {            // block column kb: TX pivot steps, then the tile shifts left
        const int k0 = kb * TX;
        const int steps = N - k0 < TX ? N - k0 : TX;
        switch (N / TX - kb + 1) {                           // live local columns
          GFR_LIVE_CASE(1) GFR_LIVE_CASE(2) GFR_LIVE_CASE(3) GFR_LIVE_CASE(4) GFR_LIVE_CASE(5)
          GFR_LIVE_CASE(6) GFR_LIVE_CASE(7) GFR_LIVE_CASE(8) GFR_LIVE_CASE(9) GFR_LIVE_CASE(10)
          default: break;
        }
        if (steps == TX) {
#pragma unroll
          for (int r = 0; r < R; ++r) {
#pragma unroll
            for (int c = 0; c + 1 < C; ++c) a[r][c] = a[r][c + 1];
            a[r][C - 1] = 0.0;
          }
        }
      }
      if (!ok) { iterations = it + 1; break; }
      __syncthreads();                                       // kof / piv of the last step; J and rhs are free
      for (int q = tid; q < ld * N; q += nt) J[q] = 0.0;     // for the next assembly pass
      if (tx == N % TX) {                                    // the right-hand-side column is local column 0 by now
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const int row = r * TY + ty;
          if (row < N) rhs[bx.kof[row]] = a[r][0] / bx.piv[row];
        }
      }
      __syncthreads();
      dense_polar_update(net, ef, rhs, accel, tid, nt);
    }
    dense_results(net, ef, red, o, env, converged, iterations, max_mismatch, tid, nt);
  }
}
template <int TX, int R>
__global__ void __launch_bounds__(8 * TX, dense_reg_min_blocks(TX, R))
dense_solve_reg_kernel(const NetDev net, const double tol, const int max_it, const double accel,
                       const double* __restrict__ p_inj, const SolOut o, const long long B) {
  dense_solve_reg<TX, R, false>(net, tol, max_it, accel, p_inj, nullptr, o, B);
}
template <int TX, int R>
__global__ void __launch_bounds__(8 * TX, dense_reg_min_blocks(TX, R))
dense_solve_reg_pq_kernel(const NetDev net, const double tol, const int max_it, const double accel,
                          const double* __restrict__ p_inj, const double* __restrict__ q_inj, const SolOut o,
                          const long long B) {
  dense_solve_reg<TX, R, true>(net, tol, max_it, accel, p_inj, q_inj, o, B);
}
#undef GFR_LIVE_CASE

#endif  // __CUDACC__

}  // namespace gfr
