// bdf_batch.cu — batched variable-order BDF integrator (orders 1-5, quasi-constant step, NDF coefficients) for sediment
// columns: the device counterpart of the reference's multistep implicit solvers.
//
// Replaces `scipy.integrate.solve_ivp(eq.fun_numba, ..., method="BDF", jac_sparsity=...)` (marlpde/parameters.py:213-216,
// :235-236; call site Evolve_scenario.py:104-109) step for step — algorithm: scipy/integrate/_ivp/bdf.py `BDF._step_impl`,
// `solve_bdf_system`, `change_D`, `BdfDenseOutput` — and is the device path for `method="LSODA"` batches (parameters.py:
// 214-219): on this stiff, diffusion-dominated system LSODA leaves its Adams mode within the first few steps and then IS
// a variable-order BDF code (measured with odeint's `mused` on the oracle: tests/test_oracle_golden.py::
// test_lsoda_runs_in_bdf_mode); its banded Jacobian with lband = uband = 1 on the field-major vector drops every
// coupling between fields, the block-tridiagonal Jacobian used here is the exact structure.
//
// Same semantics as bdf.py: differences array D[0..order+2], predictor sum(D), psi, simplified Newton (NEWTON_MAXITER = 4)
// with the same convergence-rate tests, error = error_const[order] d, the stale-LU-after-rejection policy, order selection
// from the three error norms after order+1 equal steps, step-size factors in [0.2, 10], Jacobian refreshed only after a
// Newton failure, dense output from D for t_eval and event location.  What differs is the linear algebra (shared with the
// Radau kernel, implicit_common.cuh): one warp per column, block-tridiagonal Jacobian with analytic off-diagonal blocks,
// two-ended block-Thomas factorisation of (I/c - J) in fp64, fp32 inverse Schur complements applied in the Newton sweeps
// (they only precondition the iteration: the residual c f(y) - psi - d is fp64, and the error estimate is the converged
// correction d itself, so — unlike Radau's — it carries no fp32 error).
// A resumed column (step budget) restarts at order 1 from its stored state: the differences array is not kept.
//
// kSens = true adds forward parameter sensitivities s_k = dy/d eps_k (staggered direct method, DESIGN.md 5.4): after the
// state's step is accepted every direction k takes the same NDF step for s_k' = J(y) s_k + F_k(y), with the step's order,
// h, c and the state's factors; sensitivities never enter the error test, the order selection or the step size, so the
// state's path is bit-identical with and without them.  kSens = false compiles to the kernel without sensitivities.
#include <type_traits>

#include "implicit_common.cuh"
#include "bdf_batch.cuh"

namespace marlpde {
namespace bd {
using namespace imp;

constexpr int kMaxOrder = 5;
constexpr int kNewtonMaxIter = 4;
constexpr double kMinFactor = 0.2, kMaxFactor = 10.0;
// bdf.py __init__: kappa = [0, -0.1850, -1/9, -0.0823, -0.0415, 0], gamma = [0, cumsum(1/j)], alpha = (1 - kappa) gamma,
// error_const = kappa gamma + 1/(j + 1)
__constant__ double kGamma[6] = {0.0, 1.0, 1.5, 1.8333333333333333, 2.083333333333333, 2.283333333333333};
__constant__ double kAlpha[6] = {0.0, 1.185, 1.6666666666666667, 1.9842166666666667, 2.1697916666666663, 2.283333333333333};
__constant__ double kErrConst[6] = {1.0, 0.315, 0.16666666666666666, 0.09911666666666669, 0.11354166666666668,
                                    0.16666666666666666};

// per-column workspace in doubles (n = 5 N), all vectors CELL-major [cell][field]:
//   D[8][n] | y[n] | psi[n] | d[n] | f[n] | b[n] | tmp[n] | Jacobian scratch [2n] | J [N][3][5][5] (+N) | Rec [N][128] fp32
__host__ __device__ inline size_t work_doubles(int N) {
  const size_t n = 5 * (size_t)N;
  return 16 * n + 76 * (size_t)N + 64 * (size_t)N;
}

// change_D (bdf.py): D[:order+1] <- (R U)^T D[:order+1] with R = compute_R(order, factor), U = compute_R(order, 1);
// R[i][j] = prod_{k=1..i} (k - 1 - factor j) / k.  The 6 x 6 matrices are formed by the warp in shared memory.
__device__ __noinline__ void change_D(WarpScratch& ws, int n, int lane, double* D, int order, double factor) {
  double* const R = ws.cd[0];
  double* const U = ws.cd[1];
  double* const RU = ws.cd[2];
#pragma unroll 1
  for (int e = lane; e < 36; e += 32) {
    const int i = e / 6, j = e - 6 * i;
    double r = 1.0, u = 1.0;
    for (int k = 1; k <= i; ++k) {
      r *= ((double)(k - 1) - factor * (double)j) / (double)k;
      u *= (double)(k - 1 - j) / (double)k;
    }
    R[e] = r;
    U[e] = u;
  }
  __syncwarp();
#pragma unroll 1
  for (int e = lane; e < 36; e += 32) {
    const int i = e / 6, j = e - 6 * i;
    double s = 0.0;
    for (int k = 0; k <= order; ++k) s = fma(R[i * 6 + k], U[k * 6 + j], s);
    RU[e] = s;
  }
  __syncwarp();
#pragma unroll 1
  for (int idx = lane; idx < n; idx += 32) {
    double dk[6], out[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) dk[k] = k <= order ? D[(size_t)k * n + idx] : 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < 6; ++k) s = fma(RU[k * 6 + i], dk[k], s);   // (rows k > order of dk are zero)
      out[i] = s;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i)
      if (i <= order) D[(size_t)i * n + idx] = out[i];
  }
  __syncwarp();
}

// BdfDenseOutput._call_impl at one time te: out = D[0] + sum_j D[j] prod_{m<j} (te - (t - h m)) / (h (1 + m))
__device__ __forceinline__ void dense_coeffs(double te, double t, double h, int order, double (&p)[kMaxOrder]) {
  double acc = 1.0;
#pragma unroll
  for (int m = 0; m < kMaxOrder; ++m) {
    acc *= (te - (t - h * (double)m)) / (h * (double)(1 + m));
    p[m] = m < order ? acc : 0.0;
  }
}
__device__ __forceinline__ double dense_value(const double* D, int n, int idx, int order, const double (&p)[kMaxOrder]) {
  double v = 0.0;
#pragma unroll
  for (int j = 1; j <= kMaxOrder; ++j)
    if (j <= order) v = fma(D[(size_t)j * n + idx], p[j - 1], v);
  return D[idx] + v;
}

// brentq on the dense output between t_old and t for every monitor in `act` (ivp.py handle_events): the interpolated
// state goes through a scratch vector, events are rare.
__device__ __noinline__ void locate_events(const Args& A, const ColumnConsts& kc, const fm::Tables& tb, int N, int lane,
                                           int col, unsigned act, double t_old, double t, double h, int order,
                                           const double* D, double* tmp) {
  const int n = 5 * N;
#pragma unroll 1
  for (int k = 0; k < 7; ++k) {
    if (!((act >> k) & 1u)) continue;
    BrentState bs;
    bs.init(t_old, t);
    double xeval = t_old, root = t;
    for (;;) {
      double p[kMaxOrder];
      dense_coeffs(xeval, t, h, order, p);
#pragma unroll 1
      for (int idx = lane; idx < n; idx += 32) tmp[idx] = dense_value(D, n, idx, order, p);
      __syncwarp();
      double gv[7];
      monitors(kc, tb, N, lane, tmp, nullptr, 0.0, gv);
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

// THE one instance of the RHS in this kernel, fused with the Newton residual: out = Mc f(yy) - Ml (psi + d) — the right-
// hand side M_lu (c f - psi - d) of solve_bdf_system's linear system in the scaling of factorise() — so f never travels
// through memory (Mc = 1, Ml = 0 gives the plain f(yy)).  Returns whether every lane's rates were finite.
template <bool VD>
__device__ __noinline__ bool rhs_residual(const ColumnConsts* kc, const fm::Tables* tb, int N, int lane, const double* yy,
                                          const double* psi, const double* d, double Mc, double Ml, double* out,
                                          double (*stage)[2][kStageDoubles + 6]) {
  bool finite = true;
  auto sink = [&](int i, const double (&r5)[5]) {
#pragma unroll
    for (int f = 0; f < 5; ++f) {
      finite = finite && isfinite(r5[f]);
      out[i * 5 + f] = fma(Mc, r5[f], -Ml * (psi[i * 5 + f] + d[i * 5 + f]));
    }
  };
  rhs_column<VD>(*kc, *tb, N, lane, yy, nullptr, stage, sink);
  __syncwarp();
  return __all_sync(0xffffffffu, finite);
}

// ---- forward sensitivities (kSens) ------------------------------------------------------------------------------------
// Kernel arguments of the sensitivity build: the state's arguments plus, per column c and direction k < n_dirs,
//   g_params_pm [B][P][2]   the column's parameters moved by +sigma_k / -sigma_k along direction k (host-derived)
//   g_inv2sigma [B][P]      1 / (2 sigma_k): F_k = (f(y; p+) - f(y; p-)) inv2sigma
//   g_atol_s    [B][P]      absolute tolerance of s_k in the corrector's convergence test
//   g_sens      [B][P][5][N] in: s_k at the start time (w_k); out: s_k at the time reached (field-major like y)
//   g_sens_snap [B][P][n_eval][5][N]  s_k at t_eval (field-major like the state's snapshots)
//   g_sens_stats [B][3]     accumulated: corrector iterations, fallback factorisations, unconverged steps
//   g_sens_work             sens_work_doubles(N, P) doubles per column
struct SensArgs : Args {
  const marlpde_column_params* g_params_pm;
  const double* g_inv2sigma;
  const double* g_atol_s;
  double* g_sens;
  double* g_sens_snap;
  int64_t* g_sens_stats;
  double* g_sens_work;
  int n_dirs;
};

// per-column sensitivity workspace in doubles (n = 5 N), vectors CELL-major:
//   J_s [N][3][5][5] (+N) | Rec_s [N][128] fp32 | per direction: D_s[8][n] | s[n] | psi_s[n] | d_s[n] | F[n]
__host__ __device__ inline size_t sens_work_doubles(int N, int P) {
  const size_t n = 5 * (size_t)N;
  return 76 * (size_t)N + 64 * (size_t)N + (size_t)P * 12 * n;
}

// the perturbed constants of one warp (lane 0 derives them from p+ or p-; kSens builds only)
__device__ __forceinline__ ColumnConsts* sens_consts(int warp) {
  __shared__ ColumnConsts kc_pert[kWarpsPerCta];
  return &kc_pert[warp];
}

// One RHS evaluation for the sensitivities: diff = false: out = f(yy); diff = true: out = (out - f(yy)) scale.
template <bool VD>
__device__ __noinline__ void sens_rhs(const ColumnConsts* kc, const fm::Tables* tb, int N, int lane, const double* yy,
                                      double* out, bool diff, double scale, double (*stage)[2][kStageDoubles + 6]) {
  auto sink = [&](int i, const double (&r5)[5]) {
#pragma unroll
    for (int f = 0; f < 5; ++f) out[i * 5 + f] = diff ? (out[i * 5 + f] - r5[f]) * scale : r5[f];
  };
  rhs_column<VD>(*kc, *tb, N, lane, yy, nullptr, stage, sink);
  __syncwarp();
}

// fp64 block-tridiagonal mat-vec with the Jacobian blocks of jacobian(): out = a (J x + F) - m (p + q)  (p, q may be
// NULL: then out = a (J x + F)).  One vector entry per lane and trip.
__device__ __noinline__ void sens_matvec(int N, int lane, const double* J, const double* x, const double* F, double a,
                                         double m, const double* p, const double* q, double* out) {
  const int n = 5 * N;
#pragma unroll 1
  for (int idx = lane; idx < n; idx += 32) {
    const int i = idx / 5, r = idx - 5 * i;
    const double* blk = J + (size_t)i * 75;
    double acc = F[idx];
#pragma unroll
    for (int f = 0; f < 5; ++f) acc = fma(blk[25 + f * 5 + r], x[i * 5 + f], acc);
    if (i > 0) {
#pragma unroll
      for (int f = 0; f < 5; ++f) acc = fma(blk[f * 5 + r], x[(i - 1) * 5 + f], acc);
    }
    if (i < N - 1) {
#pragma unroll
      for (int f = 0; f < 5; ++f) acc = fma(blk[50 + f * 5 + r], x[(i + 1) * 5 + f], acc);
    }
    out[idx] = p ? fma(a, acc, -m * (p[idx] + q[idx])) : a * acc;
  }
  __syncwarp();
}

// Per-column view of the sensitivity workspace.
struct SensCol {
  double* Js;
  float* Recs;
  double* dirs;
  size_t n;
  __device__ double* D(int k) const { return dirs + (size_t)k * 12 * n; }
  __device__ double* s(int k) const { return D(k) + 8 * n; }
  __device__ double* psi(int k) const { return D(k) + 9 * n; }
  __device__ double* d(int k) const { return D(k) + 10 * n; }
  __device__ double* F(int k) const { return D(k) + 11 * n; }
};

// J_s = J(yy) (the kind the column's `jac` setting selects; the finite-difference kind needs f = f(yy) with the column's
// own constants: given, or formed in ftmp when f is NULL) and F_k(yy) of every direction.  Nothing of the state is
// touched: `scratch` (2 n) is the state's Jacobian scratch and `ftmp` (n) its tmp vector, both dead between steps.
template <bool VD, bool kJacFD>
__device__ __forceinline__ void sens_prepare(WarpScratch& ws, const ColumnConsts& kc, const fm::Tables& tb, int N, int lane,
                                          const SensArgs& A, int col, const SensCol& sc, const double* yy,
                                          const double* f, double* ftmp, double* scratch) {
  if (kJacFD && !f) {
    sens_rhs<VD>(&kc, &tb, N, lane, yy, ftmp, false, 1.0, ws.stage);
    f = ftmp;
  }
  imp::jacobian<VD, kJacFD>(kc, tb, N, lane, yy, f, A.opt.atol, sc.Js, scratch, ws.stage);
  ColumnConsts* const kp = sens_consts(threadIdx.x >> 5);
#pragma unroll 1
  for (int k = 0; k < A.n_dirs; ++k) {
    const marlpde_column_params* pm = A.g_params_pm + ((size_t)col * A.n_dirs + k) * 2;
    if (lane == 0) make_consts(pm[0], N, *kp);
    __syncwarp();
    sens_rhs<VD>(kp, &tb, N, lane, yy, sc.F(k), false, 1.0, ws.stage);
    if (lane == 0) make_consts(pm[1], N, *kp);
    __syncwarp();
    sens_rhs<VD>(kp, &tb, N, lane, yy, sc.F(k), true, A.g_inv2sigma[(size_t)col * A.n_dirs + k], ws.stage);
  }
}

// The sensitivity corrector of one accepted step (order, c; the state's factors Rec hold M_lu I - J_old).  Per direction:
// s_pred = sum D_s[0..order], psi_s = D_s[1..order]^T gamma / alpha, then d_s = c (J_s s + F) - psi_s solved by the
// state's simplified Newton iteration on its own (stale) factors; if that does not converge, (I/c - J_s) is factorised
// into Rec_s once per step and the iteration restarts from the predictor; a direction that still fails keeps its last
// iterate and the step is counted as unconverged.  Leaves s_new in s, the converged correction in d_s.  `b` (n) is the
// state's right-hand-side buffer, dead between steps.
__device__ __noinline__ void sens_correct(WarpScratch& ws, int N, int lane, const SensArgs& A, int col, const SensCol& sc,
                                          int order, double c, double M_lu, const float* Rec, double newton_tol,
                                          double* b, long long& n_iter, long long& n_fact, long long& n_unconv) {
  const int n = 5 * N;
  const double rtol = A.opt.rtol;
  const double ia = 1.0 / kAlpha[order];
  bool factored = false, unconverged = false;
#pragma unroll 1
  for (int k = 0; k < A.n_dirs; ++k) {
    double* const Ds = sc.D(k);
    double* const s = sc.s(k);
    double* const psi = sc.psi(k);
    double* const d = sc.d(k);
    const double atol_s = A.g_atol_s[(size_t)col * A.n_dirs + k];
    auto predict = [&]() {
#pragma unroll 1
      for (int idx = lane; idx < n; idx += 32) {
        double v = Ds[idx], ps = 0.0;
#pragma unroll
        for (int j = 1; j <= kMaxOrder; ++j)
          if (j <= order) {
            const double x = Ds[(size_t)j * n + idx];
            v += x;
            ps = fma(x, kGamma[j], ps);
          }
        s[idx] = v;
        psi[idx] = ps * ia;
        d[idx] = 0.0;
      }
      __syncwarp();
    };
    // the state's iteration and rate test (solve_bdf_system), scale atol_s + rtol |s_pred|
    auto iterate = [&](const float* R, double Mlu) -> bool {
      const double Mc = Mlu * c;
      double norm_old = -1.0;
#pragma unroll 1
      for (int it = 0; it < kNewtonMaxIter; ++it) {
        sens_matvec(N, lane, sc.Js, s, sc.F(k), Mc, Mlu, psi, d, b);
        solve<true>(ws, N, lane, R, b, nullptr, nullptr, false);
        double ss = 0.0;
#pragma unroll 1
        for (int idx = lane; idx < n; idx += 32) {
          const double dx = b[idx], sv = s[idx], dv = d[idx];
          const double a = dx / fma(fabs(sv - dv), rtol, atol_s);
          ss = fma(a, a, ss);
          s[idx] = sv + dx;
          d[idx] = dv + dx;
        }
        __syncwarp();
        n_iter += 1;
        const double norm = sqrt(warp_sum(ss) / (double)n);
        const double rate = norm_old >= 0.0 ? norm / norm_old : -1.0;
        double rate_pow = rate;
        for (int e = 1; e < kNewtonMaxIter - it; ++e) rate_pow *= rate;
        if (!(norm == norm)) return false;
        if (rate >= 0.0 && (rate >= 1.0 || rate_pow / (1.0 - rate) * norm > newton_tol)) return false;
        if (norm == 0.0 || (rate >= 0.0 && rate / (1.0 - rate) * norm < newton_tol)) return true;
        norm_old = norm;
      }
      return false;
    };
    predict();
    if (iterate(Rec, M_lu)) continue;
    if (!factored) {
      factorise<false>(ws, N, lane, 1.0 / c, make_double2(0.0, 0.0), sc.Js, sc.Recs);
      factored = true;
      n_fact += 1;
    }
    predict();
    if (!iterate(sc.Recs, 1.0 / c)) unconverged = true;
  }
  if (unconverged) n_unconv += 1;
}

// bdf.py's post-acceptance update of the differences, applied to every D_s: D[order+2] = d - D[order+1],
// D[order+1] = d, D[i] += D[i+1] for i = order .. 0
__device__ __noinline__ void sens_update_D(int N, int lane, const SensCol& sc, int P, int order) {
  const int n = 5 * N;
#pragma unroll 1
  for (int k = 0; k < P; ++k) {
    double* const D = sc.D(k);
    const double* const d = sc.d(k);
#pragma unroll 1
    for (int idx = lane; idx < n; idx += 32) {
      const double dv = d[idx];
      D[(size_t)(order + 2) * n + idx] = dv - D[(size_t)(order + 1) * n + idx];
      D[(size_t)(order + 1) * n + idx] = dv;
      double run = dv;
#pragma unroll
      for (int i = kMaxOrder; i >= 0; --i)
        if (i <= order) {
          run += D[(size_t)i * n + idx];
          D[(size_t)i * n + idx] = run;
        }
    }
  }
  __syncwarp();
}

// every change_D of the state is applied with the same factor to every D_s
__device__ __noinline__ void sens_change_D(WarpScratch& ws, int n, int lane, const SensCol& sc, int P, int order,
                                           double factor) {
#pragma unroll 1
  for (int k = 0; k < P; ++k) change_D(ws, n, lane, sc.D(k), order, factor);
}

// resident CTAs per SM (r02v, 4096 / 64 lattice columns to t = 0.05): 2 -> 2.40 / 0.73 s, 3 -> 1.90 / 0.75 s, 4 -> 1.83 / 0.84 s
#ifndef MARLPDE_BDF_MINBLOCKS
#define MARLPDE_BDF_MINBLOCKS 3
#endif

template <bool VD, bool kJacFD, bool kSens = false>
__global__ void __launch_bounds__(kWarpsPerCta * 32, MARLPDE_BDF_MINBLOCKS)
    bdf_kernel(const std::conditional_t<kSens, SensArgs, Args> A) {
  __shared__ __align__(16) unsigned char tab_raw[fm::kTableBytes];
  __shared__ WarpScratch scratch[kWarpsPerCta];
  const fm::Tables tb = fm::stage_tables(tab_raw, threadIdx.x, blockDim.x);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  WarpScratch& ws = scratch[threadIdx.x >> 5];
  const int N = A.N, n = 5 * N;
  const double rtol = A.opt.rtol, atol = A.opt.atol;
  const double newton_tol = fmax(10.0 * kEps / rtol, fmin(0.03, sqrt(rtol)));

  for (;;) {
    int col = 0;
    if (lane == 0) col = atomicAdd(A.g_queue, 1);
    col = __shfl_sync(0xffffffffu, col, 0);
    if (col >= A.n_columns) break;

    double* const gy = A.g_y + (size_t)col * n;
    double* wbase = A.g_work + (size_t)col * work_doubles(N);
    double* const D = wbase;        wbase += 8 * (size_t)n;
    double* const y = wbase;        wbase += n;
    double* const psi = wbase;      wbase += n;
    double* const d = wbase;        wbase += n;
    double* const f = wbase;        wbase += n;
    double* const b = wbase;        wbase += n;
    double* const tmp = wbase;      wbase += n;
    double* const jscr = wbase;     wbase += 2 * (size_t)n;
    double* const J = wbase;        wbase += 76 * (size_t)N;
    float* const Rec = reinterpret_cast<float*>(wbase);
    if (lane == 0) make_consts(A.g_params[col], N, ws.kc);
#pragma unroll 1
    for (int idx = lane; idx < n; idx += 32) {
      const double v = gy[(idx % 5) * N + idx / 5];
      y[idx] = v;
      D[idx] = v;
      psi[idx] = 0.0;
      d[idx] = 0.0;
    }
    __syncwarp();
    const ColumnConsts& kc = ws.kc;
    marlpde_column_state st = A.g_state[col];
    double t = st.t, h_abs = st.h_abs;
    long long n_acc = st.n_accepted, n_rej = st.n_rejected, nfev = st.nfev;
    long long njev = 0, nlu = 0, n_newton = 0, n_newton_fail = 0;
    int next_eval = st.next_eval;
    SensCol sc{};                                        // kSens: this column's sensitivity workspace
    long long s_iter = 0, s_fact = 0, s_unconv = 0;
    const double t_start = st.t;
    if constexpr (kSens) {
      double* sb = A.g_sens_work + (size_t)col * sens_work_doubles(N, A.n_dirs);
      sc.Js = sb;
      sc.Recs = reinterpret_cast<float*>(sb + 76 * (size_t)N);
      sc.dirs = sb + 140 * (size_t)N;
      sc.n = (size_t)n;
#pragma unroll 1
      for (int k = 0; k < A.n_dirs; ++k) {
        const double* w = A.g_sens + ((size_t)col * A.n_dirs + k) * n;
        double* const Ds = sc.D(k);
        double* const s = sc.s(k);
#pragma unroll 1
        for (int idx = lane; idx < n; idx += 32) {
          const double v = w[(idx % 5) * N + idx / 5];
          s[idx] = v;
          Ds[idx] = v;
        }
      }
      __syncwarp();
    }
    int status = MARLPDE_STATUS_FINISHED;
    long long steps_done = 0;
    int order = 1, n_equal_steps = 0;
    bool lu_valid = false;
    double M_lu = 0.0;                                   // 1/c of the factors in Rec

    auto eval_to = [&](const double* yy, double* out) {   // out = f(yy)   (psi, d are finite: zeroed at column set-up)
      rhs_residual<VD>(&kc, &tb, N, lane, yy, psi, d, 1.0, 0.0, out, ws.stage);
    };
    auto jacobian = [&](const double* yy) {              // J at yy (finite-difference build: num_jac with its own f0)
      if (kJacFD) {
        eval_to(yy, tmp);
        nfev += 1 + jac_rhs_evals<kJacFD>();
      }
      imp::jacobian<VD, kJacFD>(kc, tb, N, lane, yy, tmp, atol, J, jscr, ws.stage);
      njev += 1;
    };

    if (t < A.opt.t_bound) {
      eval_to(y, f);
      nfev += 1;
      jacobian(y);
#pragma unroll 1
      for (int idx = lane; idx < n; idx += 32) D[(size_t)n + idx] = f[idx] * h_abs;   // D[1] = f h
      __syncwarp();
      if constexpr (kSens) {                             // D_s[1] = h (J(y0) w + F(y0))
        sens_prepare<VD, kJacFD>(ws, kc, tb, N, lane, A, col, sc, y, f, tmp, jscr);
#pragma unroll 1
        for (int k = 0; k < A.n_dirs; ++k)
          sens_matvec(N, lane, sc.Js, sc.s(k), sc.F(k), h_abs, 0.0, nullptr, nullptr, sc.D(k) + n);
      }
    }
    const bool ev_on = (A.opt.flags & MARLPDE_FLAG_EVENTS) != 0;
    unsigned ev_prev = 0u;
    if (ev_on && t < A.opt.t_bound) ev_prev = monitor_bits(kc, tb, N, lane, y);

    while (t < A.opt.t_bound) {
      if (A.opt.max_steps > 0 && steps_done >= A.opt.max_steps) {
        status = MARLPDE_STATUS_STEP_BUDGET;
        break;
      }
      // ------------------------------------------------------------------ bdf.py _step_impl
      const double min_step = 10.0 * (__longlong_as_double(__double_as_longlong(t) + 1) - t);
      if (h_abs > A.opt.max_step) {
        change_D(ws, n, lane, D, order, A.opt.max_step / h_abs);
        if constexpr (kSens) sens_change_D(ws, n, lane, sc, A.n_dirs, order, A.opt.max_step / h_abs);
        h_abs = A.opt.max_step;
        n_equal_steps = 0;
      } else if (h_abs < min_step) {
        change_D(ws, n, lane, D, order, min_step / h_abs);
        if constexpr (kSens) sens_change_D(ws, n, lane, sc, A.n_dirs, order, min_step / h_abs);
        h_abs = min_step;
        n_equal_steps = 0;
      }
      bool current_jac = false, accepted = false, failed = false;
      double t_new = t, safety = 1.0, error_norm = 0.0;
      int n_iter = 0;
      while (!accepted) {
        if (h_abs < min_step) {
          failed = true;
          break;
        }
        double h = h_abs;
        t_new = t + h;
        if (t_new - A.opt.t_bound > 0.0) {
          t_new = A.opt.t_bound;
          change_D(ws, n, lane, D, order, fabs(t_new - t) / h_abs);
          if constexpr (kSens) sens_change_D(ws, n, lane, sc, A.n_dirs, order, fabs(t_new - t) / h_abs);
          n_equal_steps = 0;
          lu_valid = false;
        }
        h = t_new - t;
        h_abs = fabs(h);
        const double c = h / kAlpha[order];

        bool converged = false;
        for (;;) {
          if (!lu_valid) {
            M_lu = 1.0 / c;
            factorise<false>(ws, N, lane, M_lu, make_double2(0.0, 0.0), J, Rec);
            nlu += 1;
            lu_valid = true;
          }
          // ---- y_predict = sum(D[:order+1]), psi = D[1:order+1]^T gamma[1:order+1] / alpha[order], d = 0
          {
            const double ia = 1.0 / kAlpha[order];
            _Pragma("unroll 1") for (int idx = lane; idx < n; idx += 32) {
              double s = D[idx], ps = 0.0;
#pragma unroll
              for (int k = 1; k <= kMaxOrder; ++k)
                if (k <= order) {
                  const double v = D[(size_t)k * n + idx];
                  s += v;
                  ps = fma(v, kGamma[k], ps);
                }
              y[idx] = s;
              psi[idx] = ps * ia;
              d[idx] = 0.0;
            }
            __syncwarp();
          }
          // ---- solve_bdf_system
          const double Mc = M_lu * c;                    // (I - c_lu J)^{-1} v = M_lu (M_lu I - J)^{-1} v: stale factors keep their c
          double dy_norm_old = -1.0, rate = -1.0;
          int k = 0;
          bool predict_invalid = false;                  // f(y_predict) itself is not finite
          for (k = 0; k < kNewtonMaxIter; ++k) {
            const bool finite = rhs_residual<VD>(&kc, &tb, N, lane, y, psi, d, Mc, M_lu, b, ws.stage);   // b = M_lu (c f - psi - d)
            nfev += 1;
            if (!finite) {
              predict_invalid = k == 0;
              break;
            }
            solve<true>(ws, N, lane, Rec, b, nullptr, nullptr, false);
            // norm(dy / scale) with scale = atol + rtol |y_predict| (y_predict = y - d), and in the same pass y += dy,
            // d += dy (bdf.py leaves them untouched when the rate test below breaks; they are dead then)
            double ss = 0.0;
            _Pragma("unroll 1") for (int idx = lane; idx < n; idx += 32) {
              const double dy = b[idx], yv = y[idx], dv = d[idx];
              const double a = dy / fma(fabs(yv - dv), rtol, atol);
              ss = fma(a, a, ss);
              y[idx] = yv + dy;
              d[idx] = dv + dy;
            }
            __syncwarp();
            const double dy_norm = sqrt(warp_sum(ss) / (double)n);
            rate = dy_norm_old >= 0.0 ? dy_norm / dy_norm_old : -1.0;
            double rate_pow = rate;                      // rate ** (NEWTON_MAXITER - k)
            for (int e = 1; e < kNewtonMaxIter - k; ++e) rate_pow *= rate;
            if (rate >= 0.0 && (rate >= 1.0 || rate_pow / (1.0 - rate) * dy_norm > newton_tol)) break;
            if (dy_norm == 0.0 || (rate >= 0.0 && rate / (1.0 - rate) * dy_norm < newton_tol)) {
              converged = true;
              break;
            }
            dy_norm_old = dy_norm;
          }
          n_iter = (k < kNewtonMaxIter ? k : kNewtonMaxIter - 1) + 1;
          n_newton += n_iter;
          if (converged) break;
          n_newton_fail += 1;
          if (current_jac) break;
          // bdf.py evaluates J = self.jac(t_new, y_predict) here.  ONE deliberate difference: when the predictor itself has
          // left the model's domain (extrapolated porosity <= 0: log(Phi) is NaN) that Jacobian is NaN, stays "current"
          // for the rest of the step and every smaller step size fails on it until the step size underflows (r02t: 87 of
          // 4096 lattice columns stalled this way; SciPy's own BDF has the same trap).  The step size is halved instead and
          // the Jacobian is refreshed at a predictor that can be evaluated.
          if (predict_invalid) break;
          _Pragma("unroll 1") for (int idx = lane; idx < n; idx += 32) {
            double s = D[idx];
#pragma unroll
            for (int kk = 1; kk <= kMaxOrder; ++kk)
              if (kk <= order) s += D[(size_t)kk * n + idx];
            y[idx] = s;
          }
          __syncwarp();
          jacobian(y);
          current_jac = true;
          lu_valid = false;
        }
        if (!converged) {
          h_abs *= 0.5;
          change_D(ws, n, lane, D, order, 0.5);
          if constexpr (kSens) sens_change_D(ws, n, lane, sc, A.n_dirs, order, 0.5);
          n_equal_steps = 0;
          lu_valid = false;
          continue;
        }
        safety = 0.9 * (2 * kNewtonMaxIter + 1) / (double)(2 * kNewtonMaxIter + n_iter);
        {
          const double ec = kErrConst[order];
          double ss = 0.0;
          _Pragma("unroll 1") for (int idx = lane; idx < n; idx += 32) {
            const double a = ec * d[idx] / fma(fabs(y[idx]), rtol, atol);
            ss = fma(a, a, ss);
          }
          error_norm = sqrt(warp_sum(ss) / (double)n);
        }
        if (!(error_norm <= 1.0)) {                      // (a NaN norm rejects the step; bdf.py would accept it)
          const double factor = fmax(kMinFactor, safety * pow(error_norm, -1.0 / (double)(order + 1)));
          h_abs *= factor;
          change_D(ws, n, lane, D, order, factor);
          if constexpr (kSens) sens_change_D(ws, n, lane, sc, A.n_dirs, order, factor);
          n_equal_steps = 0;
          n_rej += 1;                                    // (no trouble with convergence: the factors are kept)
        } else {
          accepted = true;
        }
      }
      if (failed) {
        status = MARLPDE_STATUS_STEP_TOO_SMALL;
        break;
      }
      if constexpr (kSens) {                             // the sensitivities' step with this step's order, h, c, factors
        sens_prepare<VD, kJacFD>(ws, kc, tb, N, lane, A, col, sc, y, nullptr, tmp, jscr);
        sens_correct(ws, N, lane, A, col, sc, order, (t_new - t) / kAlpha[order], M_lu, Rec, newton_tol, b, s_iter,
                     s_fact, s_unconv);
        sens_update_D(N, lane, sc, A.n_dirs, order);
      }
      // ------------------------------------------------------------------ accepted step
      n_equal_steps += 1;
      const double t_old = t;
      t = t_new;
      const bool adapt = n_equal_steps >= order + 1;
      // D[order+2] = d - D[order+1]; D[order+1] = d; D[i] += D[i+1] for i = order .. 0; and, when the order is
      // up for selection, the norms of error_const[order -+ 1] D[order], D[order+2] against scale(y_new)
      double ss_m = 0.0, ss_p = 0.0;
      {
        const double ecm = order > 1 ? kErrConst[order - 1] : 0.0, ecp = order < kMaxOrder ? kErrConst[order + 1] : 0.0;
        _Pragma("unroll 1") for (int idx = lane; idx < n; idx += 32) {
          const double dv = d[idx];
          const double top = dv - D[(size_t)(order + 1) * n + idx];
          D[(size_t)(order + 2) * n + idx] = top;
          D[(size_t)(order + 1) * n + idx] = dv;
          double run = dv, d_order = 0.0;
#pragma unroll
          for (int i = kMaxOrder; i >= 0; --i)
            if (i <= order) {
              run += D[(size_t)i * n + idx];
              D[(size_t)i * n + idx] = run;
              if (i == order) d_order = run;
            }
          const double isc = 1.0 / fma(fabs(y[idx]), rtol, atol);
          const double am = ecm * d_order * isc, ap = ecp * top * isc;
          ss_m = fma(am, am, ss_m);
          ss_p = fma(ap, ap, ss_p);
        }
        __syncwarp();
      }
      if (adapt) {
        const double inf = (double)INFINITY;
        const double em = order > 1 ? sqrt(warp_sum(ss_m) / (double)n) : inf;
        const double ep = order < kMaxOrder ? sqrt(warp_sum(ss_p) / (double)n) : inf;
        // factors = error_norms ** (-1 / [order, order + 1, order + 2]); argmax takes the first maximum
        const double fm_ = pow(em, -1.0 / (double)order), f0 = pow(error_norm, -1.0 / (double)(order + 1)),
                     fp = pow(ep, -1.0 / (double)(order + 2));
        int delta = -1;
        double best = fm_;
        if (f0 > best) {
          best = f0;
          delta = 0;
        }
        if (fp > best) {
          best = fp;
          delta = 1;
        }
        order += delta;
        const double factor = fmin(kMaxFactor, safety * best);
        h_abs *= factor;
        change_D(ws, n, lane, D, order, factor);
        if constexpr (kSens) sens_change_D(ws, n, lane, sc, A.n_dirs, order, factor);
        n_equal_steps = 0;
        lu_valid = false;
      }
      n_acc += 1;
      steps_done += 1;
      // ---- events (ivp.py: after every accepted step, located on the step's dense output)
      if (ev_on) {
        const unsigned ev_new = monitor_bits(kc, tb, N, lane, y);
        unsigned act = 0u;
        if (ev_new != ev_prev || (ev_new & kEqBitsMask) != 0u) act = active_events(event_classes(ev_prev), event_classes(ev_new));
        ev_prev = ev_new;
        if (act) locate_events(A, kc, tb, N, lane, col, act, t_old, t, h_abs, order, D, tmp);
      }
      // ---- t_eval samples in (t_old, t] (t_eval[0] == t0 belongs to the first step)
      while (next_eval < A.opt.n_eval) {
        const double te = A.g_t_eval[next_eval];
        if (!(te <= t)) break;
        double p[kMaxOrder];
        dense_coeffs(te, t, h_abs, order, p);
        double* snap = A.g_snap + ((size_t)col * A.opt.n_eval + next_eval) * n;
        _Pragma("unroll 1") for (int idx = lane; idx < n; idx += 32)
          snap[(idx % 5) * N + idx / 5] = dense_value(D, n, idx, order, p);
        if constexpr (kSens) {                           // (a sample at the start time is w itself)
#pragma unroll 1
          for (int k = 0; k < A.n_dirs; ++k) {
            const double* w = A.g_sens + ((size_t)col * A.n_dirs + k) * n;
            double* ss = A.g_sens_snap + (((size_t)col * A.n_dirs + k) * A.opt.n_eval + next_eval) * n;
            const double* Ds = sc.D(k);
            _Pragma("unroll 1") for (int idx = lane; idx < n; idx += 32) {
              const int fi = (idx % 5) * N + idx / 5;
              ss[fi] = te == t_start ? w[fi] : dense_value(Ds, n, idx, order, p);
            }
          }
        }
        ++next_eval;
      }
    }
    // the state at time t: y (= y_new of the last accepted step); after a failed step y holds a Newton iterate, the
    // last accepted state is then D[0] (change_D leaves row 0 alone)
    const double* const y_out = status == MARLPDE_STATUS_STEP_TOO_SMALL ? D : y;
#pragma unroll 1
    for (int idx = lane; idx < n; idx += 32) gy[(idx % 5) * N + idx / 5] = y_out[idx];
    if constexpr (kSens) {                               // s at time t, mirroring y_out (w is read above: sync first)
      __syncwarp();
#pragma unroll 1
      for (int k = 0; k < A.n_dirs; ++k) {
        const double* s_out = status == MARLPDE_STATUS_STEP_TOO_SMALL ? sc.D(k) : sc.s(k);
        double* gs = A.g_sens + ((size_t)col * A.n_dirs + k) * n;
#pragma unroll 1
        for (int idx = lane; idx < n; idx += 32) gs[(idx % 5) * N + idx / 5] = s_out[idx];
      }
      if (lane == 0) {
        int64_t* s3 = A.g_sens_stats + (size_t)col * 3;
        s3[0] += s_iter;
        s3[1] += s_fact;
        s3[2] += s_unconv;
      }
    }
    if (lane == 0) {
      st.t = t;
      st.h_abs = h_abs;
      st.n_accepted = n_acc;
      st.n_rejected = n_rej;
      st.nfev = nfev;
      st.status = status;
      st.next_eval = next_eval;
      A.g_state[col] = st;
      int64_t* s4 = A.g_stats + (size_t)col * 4;
      s4[0] += njev;
      s4[1] += nlu;
      s4[2] += n_newton;
      s4[3] += n_newton_fail;
    }
    __syncwarp();
  }
}

}  // namespace bd

size_t bdf_workspace_bytes(int n_columns, int n_cells) {
  return sizeof(double) * bd::work_doubles(n_cells) * (size_t)n_columns;
}

#ifndef MARLPDE_HOST_EMU
cudaError_t launch_bdf(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                       int n_columns, int n_cells, const marlpde_rk45_options& opt, const double* d_t_eval,
                       double* d_snap, int64_t* d_stats, int32_t* d_ev_counts, double* d_ev_times, double* d_work,
                       int32_t* d_queue, int sm_count, cudaStream_t stream) {
  imp::Args a;
  a.g_y = d_y;
  a.g_params = d_params;
  a.g_state = d_state;
  a.g_t_eval = d_t_eval;
  a.g_snap = d_snap;
  a.g_stats = d_stats;
  a.g_ev_counts = d_ev_counts;
  a.g_ev_times = d_ev_times;
  a.g_work = d_work;
  a.g_queue = d_queue;
  a.n_columns = n_columns;
  a.N = n_cells;
  a.opt = opt;
  int ctas = (n_columns + imp::kWarpsPerCta - 1) / imp::kWarpsPerCta;
  const int max_ctas = sm_count * MARLPDE_BDF_MINBLOCKS;
  if (ctas > max_ctas) ctas = max_ctas;
  if (ctas < 1) ctas = 1;
  const bool vd = (opt.flags & MARLPDE_FLAG_VAR_DPHI) != 0, fd = (opt.flags & MARLPDE_FLAG_JAC_FD) != 0;
  const int threads = imp::kWarpsPerCta * 32;
  if (vd && fd) bd::bdf_kernel<true, true><<<ctas, threads, 0, stream>>>(a);
  else if (vd) bd::bdf_kernel<true, false><<<ctas, threads, 0, stream>>>(a);
  else if (fd) bd::bdf_kernel<false, true><<<ctas, threads, 0, stream>>>(a);
  else bd::bdf_kernel<false, false><<<ctas, threads, 0, stream>>>(a);
  return cudaGetLastError();
}
#endif

size_t bdf_sens_workspace_bytes(int n_columns, int n_cells, int n_dirs) {
  return sizeof(double) * bd::sens_work_doubles(n_cells, n_dirs) * (size_t)n_columns;
}

#ifndef MARLPDE_HOST_EMU
namespace bd {
// bad[0] += number of (column, direction, sign) whose perturbed parameters differ from the column's in an integer field
__global__ void sens_check_kernel(const marlpde_column_params* p, const marlpde_column_params* pm, int n_columns,
                                  int n_dirs, int32_t* bad) {
  const long long total = 2LL * n_columns * n_dirs;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const marlpde_column_params& a = p[e / (2 * n_dirs)];
    const marlpde_column_params& q = pm[e];
    if (a.FV_switch != q.FV_switch || a.mask_lo != q.mask_lo || a.mask_hi != q.mask_hi || a.model_flags != q.model_flags)
      atomicAdd(bad, 1);
  }
}
}  // namespace bd

cudaError_t launch_bdf_sens_check(const marlpde_column_params* d_params, const marlpde_column_params* d_params_pm,
                                  int n_columns, int n_dirs, int32_t* d_bad, cudaStream_t stream) {
  const long long total = 2LL * n_columns * n_dirs;
  const int blocks = (int)((total + 255) / 256 < 1024 ? (total + 255) / 256 : 1024);
  bd::sens_check_kernel<<<blocks > 0 ? blocks : 1, 256, 0, stream>>>(d_params, d_params_pm, n_columns, n_dirs, d_bad);
  return cudaGetLastError();
}

cudaError_t launch_bdf_sens(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                            int n_columns, int n_cells, const marlpde_rk45_options& opt, const double* d_t_eval,
                            double* d_snap, int64_t* d_stats, int32_t* d_ev_counts, double* d_ev_times, double* d_work,
                            int32_t* d_queue, int n_dirs, const marlpde_column_params* d_params_pm,
                            const double* d_inv2sigma, const double* d_atol_s, double* d_sens, double* d_sens_snap,
                            int64_t* d_sens_stats, double* d_sens_work, int sm_count, cudaStream_t stream) {
  bd::SensArgs a;
  a.g_y = d_y;
  a.g_params = d_params;
  a.g_state = d_state;
  a.g_t_eval = d_t_eval;
  a.g_snap = d_snap;
  a.g_stats = d_stats;
  a.g_ev_counts = d_ev_counts;
  a.g_ev_times = d_ev_times;
  a.g_work = d_work;
  a.g_queue = d_queue;
  a.n_columns = n_columns;
  a.N = n_cells;
  a.opt = opt;
  a.g_params_pm = d_params_pm;
  a.g_inv2sigma = d_inv2sigma;
  a.g_atol_s = d_atol_s;
  a.g_sens = d_sens;
  a.g_sens_snap = d_sens_snap;
  a.g_sens_stats = d_sens_stats;
  a.g_sens_work = d_sens_work;
  a.n_dirs = n_dirs;
  int ctas = (n_columns + imp::kWarpsPerCta - 1) / imp::kWarpsPerCta;
  const int max_ctas = sm_count * MARLPDE_BDF_MINBLOCKS;
  if (ctas > max_ctas) ctas = max_ctas;
  if (ctas < 1) ctas = 1;
  const bool vd = (opt.flags & MARLPDE_FLAG_VAR_DPHI) != 0, fd = (opt.flags & MARLPDE_FLAG_JAC_FD) != 0;
  const int threads = imp::kWarpsPerCta * 32;
  if (vd && fd) bd::bdf_kernel<true, true, true><<<ctas, threads, 0, stream>>>(a);
  else if (vd) bd::bdf_kernel<true, false, true><<<ctas, threads, 0, stream>>>(a);
  else if (fd) bd::bdf_kernel<false, true, true><<<ctas, threads, 0, stream>>>(a);
  else bd::bdf_kernel<false, false, true><<<ctas, threads, 0, stream>>>(a);
  return cudaGetLastError();
}
#endif

}  // namespace marlpde
