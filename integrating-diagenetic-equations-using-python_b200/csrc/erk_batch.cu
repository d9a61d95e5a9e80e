// erk_batch.cu — batched explicit Runge-Kutta integrators for sediment columns: Bogacki-Shampine RK23 and Dormand-Prince
// DOP853, the two `solve_ivp` methods the implicit and RK45 kernels leave out.
//
// Replaces `scipy.integrate.solve_ivp(eq.fun_numba, ..., method="RK23" | "DOP853")` (marlpde/parameters.py:213; call site
// Evolve_scenario.py:104-109) step for step — algorithm: scipy/integrate/_ivp/rk.py `rk_step`, `RungeKutta._step_impl`,
// `DOP853._estimate_error_norm`, `RkDenseOutput`, `Dop853DenseOutput`; the tableaux are generated from the installed
// SciPy's class attributes (gen_erk_tables.py -> erk_tables.inc).  One kernel template, instantiated per tableau:
//   * step control of _step_impl: SAFETY 0.9, factors in [0.2, 10], min_step = 10 ulp(t), no growth right after a
//     rejection, the last step clipped to t_bound, error exponent -1 / (error_estimator_order + 1);
//   * error norm: RK23 the RMS norm of h K^T E / scale, DOP853 its combination of the E5 and E3 estimates;
//   * dense output, for t_eval samples and event location: RK23 the cubic y_old + h sum_k (K^T P)_k x^(k+1); DOP853
//     three extra stages and seven F arrays evaluated with the nested x / (1 - x) products.  As in ivp.py the extra stages
//     are evaluated only in steps that sample a t_eval point or locate an event, and they count in nfev.
// The machinery is the implicit kernels' (implicit_common.cuh): one warp per column claimed from a queue, every vector in
// an HBM workspace (any n_cells >= 3), the one `rhs_eval` instance, `monitor_bits` after each accepted step, `monitors` +
// BrentState on the dense output for event location.
// A column that stops on its step budget stops after an accepted step; f(y) is recomputed bit-identically when it
// resumes, so a run cut into budgets equals an uninterrupted one bit for bit (nfev counts the extra evaluation).
#include "implicit_common.cuh"
#include "erk_batch.cuh"

namespace marlpde {
namespace erk {
using namespace imp;

#include "erk_tables.inc"

constexpr double kSafety = 0.9, kMinFactor = 0.2, kMaxFactor = 10.0;

// Tableaux.  kStages: stages of a step (K[0] = f(y) comes from the previous step); row kStages of K holds f(y_new);
// rows kStages + 1 .. kRows - 1 are the extra stages of the dense output.
struct RK23 {
  static constexpr int kStages = 3, kRows = 4;
  static constexpr bool kDop = false;
  static constexpr double kErrExp = -1.0 / 3.0;     // -1 / (error_estimator_order + 1), error_estimator_order = 2
  __device__ static double a(int s, int j) { return erk23::kA[s][j]; }
  __device__ static double b(int j) { return erk23::kB[j]; }
};
struct DOP853 {
  static constexpr int kStages = 12, kRows = 16;
  static constexpr bool kDop = true;
  static constexpr double kErrExp = -1.0 / 8.0;     // error_estimator_order = 7
  __device__ static double a(int s, int j) { return dop853::kA[s][j]; }
  __device__ static double b(int j) { return dop853::kB[j]; }
};

// per-column workspace in doubles (n = 5 N), all vectors CELL-major [cell][field]:  y[n] | y_new[n] | stage input[n] | K[kRows][n]
template <class M>
__host__ __device__ inline size_t work_doubles(int N) {
  return (3 + (size_t)M::kRows) * 5 * (size_t)N;
}

// Everything one column's step needs: the vectors of the workspace and the step being taken.
struct Column {
  double* y;          // state at t (y_old of the step just accepted, until it is committed)
  double* yn;         // y_new
  double* ys;         // stage input; also the dense-output state during event location
  double* K;          // kRows rows of n
  int n;
  int f0, fN;         // physical rows of K[0] = f(y) and K[kStages] = f(y_new): swapped when a step is committed (FSAL)
  __device__ double* row(int s, int kStages) const {
    const int p = s == 0 ? f0 : (s == kStages ? fN : s);
    return K + (size_t)p * n;
  }
};

// ys = y + h sum_{j<s} a_sj K_j  (rk_step: dy = K[:s].T a[:s] * h)
template <class M>
__device__ __forceinline__ void stage_input(const Column& c, int lane, int s, double h) {
#pragma unroll 1
  for (int idx = lane; idx < c.n; idx += 32) {
    double acc = 0.0;
#pragma unroll 1
    for (int j = 0; j < s; ++j) {
      const double a = M::a(s, j);
      if (a != 0.0) acc = fma(a, c.row(j, M::kStages)[idx], acc);
    }
    c.ys[idx] = c.y[idx] + acc * h;
  }
  __syncwarp();
}

// dense output of the accepted step (t_old, t_old + h) at x = (te - t_old) / h, element idx
template <class M>
__device__ __forceinline__ double dense_value(const Column& c, int idx, double x, double h) {
  const double yo = c.y[idx];
  if constexpr (!M::kDop) {
    // RkDenseOutput: Q = K^T P, y = y_old + h Q [x, x^2, x^3]
    double q[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int s = 0; s < M::kRows; ++s) {
      const double k = c.row(s, M::kStages)[idx];
#pragma unroll
      for (int j = 0; j < 3; ++j) q[j] = fma(k, erk23::kP[s][j], q[j]);
    }
    return fma(h, x * (q[0] + x * (q[1] + x * q[2])), yo);
  } else {
    // Dop853DenseOutput: F0 = dy, F1 = h f_old - dy, F2 = 2 dy - h (f_new + f_old), F3..6 = h D K;
    // y = y_old + (((((((F6 x + F5)(1-x) + F4) x + F3)(1-x) + F2) x + F1)(1-x) + F0) x
    const double f_old = c.row(0, M::kStages)[idx], f_new = c.row(M::kStages, M::kStages)[idx];
    const double dy = c.yn[idx] - yo;
    double F[7];
    F[0] = dy;
    F[1] = h * f_old - dy;
    F[2] = 2.0 * dy - h * (f_new + f_old);
#pragma unroll
    for (int r = 0; r < 4; ++r) F[3 + r] = 0.0;
#pragma unroll 1
    for (int s = 0; s < M::kRows; ++s) {
      const double k = c.row(s, M::kStages)[idx];
#pragma unroll
      for (int r = 0; r < 4; ++r) F[3 + r] = fma(dop853::kD[r][s], k, F[3 + r]);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) F[3 + r] *= h;
    const double xm = 1.0 - x;
    double v = 0.0;
#pragma unroll
    for (int i = 0; i < 7; ++i) v = (v + F[6 - i]) * ((i & 1) ? xm : x);
    return v + yo;
  }
}

// brentq on the dense output between t_old and t for every monitor in `act` (ivp.py handle_events)
template <class M>
__device__ __noinline__ void locate_events(const Args& A, const ColumnConsts& kc, const fm::Tables& tb, int N, int lane,
                                           int col, unsigned act, double t_old, double t, double h, const Column& c) {
#pragma unroll 1
  for (int k = 0; k < 7; ++k) {
    if (!((act >> k) & 1u)) continue;
    BrentState bs;
    bs.init(t_old, t);
    double xeval = t_old, root = t;
    for (;;) {
      const double x = (xeval - t_old) / h;
#pragma unroll 1
      for (int idx = lane; idx < c.n; idx += 32) c.ys[idx] = dense_value<M>(c, idx, x, h);
      __syncwarp();
      double gv[7];
      monitors(kc, tb, N, lane, c.ys, nullptr, 0.0, gv);
      double gk = gv[0];
#pragma unroll
      for (int kk = 1; kk < 7; ++kk) gk = (k == kk) ? gv[kk] : gk;
      __syncwarp();
      if (bs.feed(gk, xeval, root)) break;
    }
    if (lane == 0) {
      int32_t* cnt = A.g_ev_counts + (size_t)col * MARLPDE_NEVENTS + k;
      const int have = *cnt;
      if (have < A.opt.event_capacity)
        A.g_ev_times[((size_t)col * MARLPDE_NEVENTS + k) * A.opt.event_capacity + have] = root;
      *cnt = have + 1;
    }
  }
}

// resident CTAs per SM the kernel is compiled for: 3 (168 registers per thread; ptxas: rhs_eval spills 16-48 bytes, the
// kernel body 384-408 bytes of stores around its calls) rather than the 4 the shared memory would allow (128 registers:
// rhs_eval spills 168-232 bytes, the kernel body 436-540).  Not measured against each other yet.
#ifndef MARLPDE_ERK_MINBLOCKS
#define MARLPDE_ERK_MINBLOCKS 3
#endif

template <class M, bool VD>
__global__ void __launch_bounds__(kWarpsPerCta * 32, MARLPDE_ERK_MINBLOCKS) erk_kernel(const Args A) {
  __shared__ __align__(16) unsigned char tab_raw[fm::kTableBytes];
  __shared__ WarpScratch scratch[kWarpsPerCta];
  const fm::Tables tb = fm::stage_tables(tab_raw, threadIdx.x, blockDim.x);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  WarpScratch& ws = scratch[threadIdx.x >> 5];
  const int N = A.N, n = 5 * N;
  const double rtol = A.opt.rtol, atol = A.opt.atol, t_bound = A.opt.t_bound;
  const double sqrt_n = sqrt((double)n);
  constexpr int S = M::kStages;

  for (;;) {
    int col = 0;
    if (lane == 0) col = atomicAdd(A.g_queue, 1);
    col = __shfl_sync(0xffffffffu, col, 0);
    if (col >= A.n_columns) break;

    double* const gy = A.g_y + (size_t)col * n;
    double* const wbase = A.g_work + (size_t)col * work_doubles<M>(N);
    Column c;
    c.y = wbase;
    c.yn = wbase + n;
    c.ys = wbase + 2 * (size_t)n;
    c.K = wbase + 3 * (size_t)n;
    c.n = n;
    c.f0 = 0;
    c.fN = S;
    if (lane == 0) make_consts(A.g_params[col], N, ws.kc);
#pragma unroll 1
    for (int idx = lane; idx < n; idx += 32) c.y[idx] = gy[(idx % 5) * N + idx / 5];
    __syncwarp();
    const ColumnConsts& kc = ws.kc;
    marlpde_column_state st = A.g_state[col];
    double t = st.t, h_abs = st.h_abs;
    long long n_acc = st.n_accepted, n_rej = st.n_rejected, nfev = st.nfev;
    int next_eval = st.next_eval;
    int status = MARLPDE_STATUS_FINISHED;
    long long attempts = 0;
    auto rhs = [&](const double* yy, double* out) { rhs_eval<VD>(&kc, &tb, N, lane, yy, nullptr, out, ws.stage); };

    const bool ev_on = (A.opt.flags & MARLPDE_FLAG_EVENTS) != 0;
    unsigned ev_prev = 0u;
    if (t < t_bound) {
      rhs(c.y, c.row(0, S));                             // self.f = fun(t0, y0)
      nfev += 1;
      if (ev_on) ev_prev = monitor_bits(kc, tb, N, lane, c.y);
    }

    while (t < t_bound) {
      if (A.opt.max_steps > 0 && attempts >= A.opt.max_steps) {
        status = MARLPDE_STATUS_STEP_BUDGET;
        break;
      }
      // ------------------------------------------------------------------ rk.py _step_impl
      const double min_step = 10.0 * fabs(nextafter(t, (double)INFINITY) - t);
      if (h_abs > A.opt.max_step) h_abs = A.opt.max_step;
      else if (h_abs < min_step) h_abs = min_step;
      bool rejected = false, failed = false;
      double t_new = t, h = 0.0;
      for (;;) {
        if (h_abs < min_step) {
          failed = true;
          break;
        }
        h = h_abs;
        t_new = t + h;
        if (t_new - t_bound > 0.0) t_new = t_bound;
        h = t_new - t;
        h_abs = fabs(h);
        // ---- rk_step: stages 1 .. S-1, y_new = y + h K[:S]^T B, K[S] = f(y_new)
#pragma unroll 1
        for (int s = 1; s < S; ++s) {
          stage_input<M>(c, lane, s, h);
          rhs(c.ys, c.row(s, S));
        }
#pragma unroll 1
        for (int idx = lane; idx < n; idx += 32) {
          double acc = 0.0;
#pragma unroll 1
          for (int j = 0; j < S; ++j) {
            const double b = M::b(j);
            if (b != 0.0) acc = fma(b, c.row(j, S)[idx], acc);
          }
          c.yn[idx] = c.y[idx] + h * acc;
        }
        __syncwarp();
        rhs(c.yn, c.row(S, S));
        nfev += S;
        attempts += 1;
        // ---- error norm against scale = atol + max(|y|, |y_new|) rtol
        double e_a = 0.0, e_b = 0.0;                     // RK23: sum (err/scale)^2; DOP853: sums of err5^2, err3^2
#pragma unroll 1
        for (int idx = lane; idx < n; idx += 32) {
          const double isc = 1.0 / fma(fmax(fabs(c.y[idx]), fabs(c.yn[idx])), rtol, atol);
          if constexpr (!M::kDop) {
            double e = 0.0;
#pragma unroll
            for (int j = 0; j <= S; ++j) e = fma(erk23::kE[j], c.row(j, S)[idx], e);
            const double q = (e * h) * isc;
            e_a = fma(q, q, e_a);
          } else {
            double e5 = 0.0, e3 = 0.0;
#pragma unroll 1
            for (int j = 0; j <= S; ++j) {
              const double c5 = dop853::kE5[j], c3 = dop853::kE3[j];
              if (c5 != 0.0 || c3 != 0.0) {
                const double k = c.row(j, S)[idx];
                e5 = fma(c5, k, e5);
                e3 = fma(c3, k, e3);
              }
            }
            e5 *= isc;
            e3 *= isc;
            e_a = fma(e5, e5, e_a);
            e_b = fma(e3, e3, e_b);
          }
        }
        double error_norm;
        if constexpr (!M::kDop) {
          error_norm = sqrt(warp_sum(e_a)) / sqrt_n;     // common.py norm: ||x|| / sqrt(x.size)
        } else {
          const double s5 = warp_sum(e_a), s3 = warp_sum(e_b);
          error_norm = (s5 == 0.0 && s3 == 0.0) ? 0.0 : fabs(h) * s5 / sqrt((s5 + 0.01 * s3) * (double)n);
        }
        if (error_norm < 1.0) {
          double factor = kMaxFactor;
          if (error_norm != 0.0) factor = fmin(kMaxFactor, kSafety * pow(error_norm, M::kErrExp));
          if (rejected) factor = fmin(1.0, factor);
          h_abs *= factor;
          break;
        }
        // NaN error norms land here too: fmax drops the NaN, like Python's max(0.2, nan)
        h_abs *= fmax(kMinFactor, kSafety * pow(error_norm, M::kErrExp));
        rejected = true;
        n_rej += 1;
      }
      if (failed) {
        status = MARLPDE_STATUS_STEP_TOO_SMALL;
        break;
      }
      // ------------------------------------------------------------------ accepted step (t_old, t]
      n_acc += 1;
      const double t_old = t;
      t = t_new;
      unsigned act = 0u, ev_new = 0u;
      if (ev_on) {
        ev_new = monitor_bits(kc, tb, N, lane, c.yn);
        if (ev_new != ev_prev || (ev_new & kEqBitsMask) != 0u) act = active_events(event_classes(ev_prev), event_classes(ev_new));
        ev_prev = ev_new;
      }
      const bool sample = next_eval < A.opt.n_eval && A.g_t_eval[next_eval] <= t;
      if constexpr (M::kDop) {
        // Dop853 _dense_output_impl, only when ivp.py asks for the step's dense output
        if (act || sample) {
#pragma unroll 1
          for (int s = S + 1; s < M::kRows; ++s) {
            stage_input<M>(c, lane, s, h);
            rhs(c.ys, c.row(s, S));
          }
          nfev += M::kRows - S - 1;
        }
      }
      if (act) locate_events<M>(A, kc, tb, N, lane, col, act, t_old, t, h, c);
      // ---- t_eval samples in (t_old, t] (t_eval[0] == t0 belongs to the first step)
      while (next_eval < A.opt.n_eval) {
        const double te = A.g_t_eval[next_eval];
        if (!(te <= t)) break;
        const double x = (te - t_old) / h;
        double* snap = A.g_snap + ((size_t)col * A.opt.n_eval + next_eval) * n;
#pragma unroll 1
        for (int idx = lane; idx < n; idx += 32) snap[(idx % 5) * N + idx / 5] = dense_value<M>(c, idx, x, h);
        ++next_eval;
      }
      __syncwarp();
      // ---- commit: y <- y_new, f <- f_new (FSAL)
      double* const tmp = c.y;
      c.y = c.yn;
      c.yn = tmp;
      const int fr = c.f0;
      c.f0 = c.fN;
      c.fN = fr;
    }
#pragma unroll 1
    for (int idx = lane; idx < n; idx += 32) gy[(idx % 5) * N + idx / 5] = c.y[idx];
    if (lane == 0) {
      st.t = t;
      st.h_abs = h_abs;
      st.n_accepted = n_acc;
      st.n_rejected = n_rej;
      st.nfev = nfev;
      st.status = status;
      st.next_eval = next_eval;
      A.g_state[col] = st;
    }
    __syncwarp();
  }
}

}  // namespace erk

size_t erk_workspace_bytes(ErkMethod method, int n_columns, int n_cells) {
  const size_t per = method == kErkRK23 ? erk::work_doubles<erk::RK23>(n_cells) : erk::work_doubles<erk::DOP853>(n_cells);
  return sizeof(double) * per * (size_t)n_columns;
}

#ifndef MARLPDE_HOST_EMU
cudaError_t launch_erk(ErkMethod method, double* d_y, const marlpde_column_params* d_params,
                       marlpde_column_state* d_state, int n_columns, int n_cells, const marlpde_rk45_options& opt,
                       const double* d_t_eval, double* d_snap, int32_t* d_ev_counts, double* d_ev_times,
                       double* d_work, int32_t* d_queue, int sm_count, cudaStream_t stream) {
  imp::Args a;
  a.g_y = d_y;
  a.g_params = d_params;
  a.g_state = d_state;
  a.g_t_eval = d_t_eval;
  a.g_snap = d_snap;
  a.g_stats = nullptr;
  a.g_ev_counts = d_ev_counts;
  a.g_ev_times = d_ev_times;
  a.g_work = d_work;
  a.g_queue = d_queue;
  a.n_columns = n_columns;
  a.N = n_cells;
  a.opt = opt;
  int ctas = (n_columns + imp::kWarpsPerCta - 1) / imp::kWarpsPerCta;
  const int max_ctas = sm_count * MARLPDE_ERK_MINBLOCKS;
  if (ctas > max_ctas) ctas = max_ctas;
  if (ctas < 1) ctas = 1;
  const bool vd = (opt.flags & MARLPDE_FLAG_VAR_DPHI) != 0;
  const int threads = imp::kWarpsPerCta * 32;
  if (method == kErkRK23) {
    if (vd) erk::erk_kernel<erk::RK23, true><<<ctas, threads, 0, stream>>>(a);
    else erk::erk_kernel<erk::RK23, false><<<ctas, threads, 0, stream>>>(a);
  } else {
    if (vd) erk::erk_kernel<erk::DOP853, true><<<ctas, threads, 0, stream>>>(a);
    else erk::erk_kernel<erk::DOP853, false><<<ctas, threads, 0, stream>>>(a);
  }
  return cudaGetLastError();
}
#endif

}  // namespace marlpde
