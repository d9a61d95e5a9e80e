// rk45_streaming.cu — adaptive Dormand-Prince 5(4) for depth grids too large for shared memory
// (BASELINE.json configs[3]: N = 2 000 ... 20 000 cells, 1-64 columns).
//
// Same stepper as rk45_persistent.cu (scipy RK45 semantics per column: rk.py `_step_impl`, `rk_step`,
// `RkDenseOutput`; call site marlpde/Evolve_scenario.py:104-109) and the same rhs_pair arithmetic, but
// a column is cut into overlapping windows and only y and the stage derivatives stream through HBM/L2:
//   * state, stage derivatives K1..K7 and a second y buffer are [column][field][cell] arrays in a
//     caller-provided workspace; an accepted step writes y_new to the y buffer not in use and flips
//     the index instead of copying;
//   * ONE launch of tile_attempt_kernel per step attempt: a CTA integrates one window of a column
//     through all six stages and the FSAL evaluation on chip (see below) and writes y_new, K7 and its
//     window's contribution to the error norm.  The kernel boundary is the only synchronisation
//     between windows, so columns never wait for each other inside a kernel;
//   * per-column control (error norm from per-window partial sums added in fixed order, accept/reject,
//     step-size factor, t_eval dense output, FSAL by swapping two slot indices instead of copying K7)
//     runs in the prologue of the next attempt's launch (close_and_begin); prepare_kernel closes the
//     last attempt of a call.  Control blocks are double buffered, so every CTA of a column derives
//     the same decision from the same inputs while the column's first CTA publishes the updated block;
//   * algorithmic HBM traffic: 4 vector passes of 40 bytes per cell and attempt = 160 B per cell
//     (DESIGN.md §4.4); the L2 keeps working sets up to ~100 MB on chip.
// A call enqueues a fixed number of step attempts (no host round trip, no synchronisation); columns
// that reach t_bound earlier idle, columns that do not come back resumable with status STEP_BUDGET.
// K1 = f(y) of the first attempt comes from k1_kernel.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "brent.cuh"
#include "dopri.cuh"
#include "events.cuh"
#include "lheureux_device.cuh"
#include "mbar.cuh"
#include "rk45_streaming.cuh"

namespace marlpde {
namespace st {

constexpr int kThreads = 128;                 // pairs per CTA
constexpr int kCellsPerCta = 2 * kThreads;

struct Ctl {                                   // per-column control block (double buffered)
  double t, h_abs, h, t_new;
  long long n_acc, n_rej, nfev, attempts;
  int status;                                  // MARLPDE_STATUS_* once inactive
  int active;                                  // 1: attempt in flight / to be started
  int rejected;                                // a rejection happened within the current step
  int next_eval;
  int k1, k7;                                  // physical slots of K1 and K7 (0 or 6)
  int fresh;                                   // 1: K1 has just been evaluated, no attempt finished yet
  int midstep;                                 // resumed inside a step (after a rejected attempt)
  int ysl;                                     // which buffer holds y (0: caller's y, 1: workspace vector 0)
  int locate;                                  // events: 1 = the accepted step in flight has a sign change; the attempt
                                               // is replayed with K3..K6 stored, then its roots are located and it commits
  unsigned ev_prev;                            // predicate bits of the monitors at the start of the current step
  int skip;                                    // the attempt described here has NOT been run yet (the launch that
                                               // located the events of the previous step ran no attempt): nothing to close
};

struct Args {
  double* y;                 // [B][5][N] state (updated in place on accepted steps)
  const marlpde_column_params* params;
  marlpde_column_state* state;
  const double* t_eval;
  double* snap;
  double* K;                 // [7][B][5][N]
  double* tile;              // [B][5][N] second y buffer (workspace vector 0)
  double* partials;          // [2][B][pstride]: written by the launch that runs an attempt under control buffer p into
                             // parity p, read by the launch that closes it (the tile kernel closes the previous
                             // attempt in its prologue while faster CTAs of the same launch already write the next sums)
  Ctl* ctl;                  // [2][B]
  unsigned* evpart;          // [2][B][pstride] predicate bits of the monitors per CTA / window (MARLPDE_FLAG_EVENTS)
  int32_t* ev_counts;        // [B][7]
  double* ev_times;          // [B][7][event_capacity]
  int B, N, tiles;
  int tiles2;                // tile_attempt_kernel windows per column
  int pstride;               // entries per column in `partials` and `evpart`
  marlpde_rk45_options opt;
};

__host__ __device__ inline size_t align256(size_t x) { return (x + 255) / 256 * 256; }

// Workspace layout (marlpde_rk45_stream_workspace_bytes).  Of the two vectors at off_tile only the first is used (the
// second y buffer); the second slot is kept so that the workspace size seen through the C ABI does not change.
struct Layout {
  size_t off_K, off_tile, off_part, off_ctl, off_ev, total;
};
__host__ inline Layout layout(int B, int N) {
  const size_t vec = sizeof(double) * 5 * (size_t)N * B;
  const int tiles = (N + 243) / 244 + 1;       // >= CTAs per column of every kernel (256-cell CTAs, 244- / 628-cell windows)
  Layout L;
  size_t o = 0;
  L.off_K = o;     o += align256(7 * vec);
  L.off_tile = o;  o += align256(2 * vec);
  L.off_part = o;  o += align256(sizeof(double) * 2 * (size_t)tiles * B);     // [2 parities][B][tiles]
  L.off_ctl = o;   o += align256(sizeof(Ctl) * 2 * (size_t)B);
  L.off_ev = o;    o += align256(sizeof(unsigned) * 2 * (size_t)tiles * B);
  L.total = o;
  return L;
}

__device__ __forceinline__ double min_step_at(double t) { return 10.0 * fabs(nextafter(t, (double)INFINITY) - t); }

// rk.py _step_impl prologue: clamp h_abs at the start of a step; then the attempt's (h, t_new)
__device__ __forceinline__ void begin_step(Ctl& c, const marlpde_rk45_options& opt) {
  const double ms = min_step_at(c.t);
  if (c.h_abs > opt.max_step) c.h_abs = opt.max_step;
  else if (c.h_abs < ms) c.h_abs = ms;
  c.rejected = 0;
}
__device__ __forceinline__ bool begin_attempt(Ctl& c, const marlpde_rk45_options& opt) {
  if (c.h_abs < min_step_at(c.t)) return false;
  double h = c.h_abs;
  c.t_new = c.t + h;
  if (c.t_new - opt.t_bound > 0.0) c.t_new = opt.t_bound;
  h = c.t_new - c.t;
  c.h = h;
  c.h_abs = fabs(h);
  return true;
}

// ---- control blocks from the caller's per-column state (one thread per column)
__global__ void init_kernel(const Args A) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= A.B) return;
  const marlpde_column_state s = A.state[col];
  Ctl c;
  c.t = s.t;
  c.h_abs = s.h_abs;
  c.h = 0.0;
  c.t_new = s.t;
  c.n_acc = s.n_accepted;
  c.n_rej = s.n_rejected;
  c.nfev = s.nfev;
  c.attempts = 0;
  c.status = MARLPDE_STATUS_STEP_BUDGET;
  c.active = 1;
  c.rejected = 0;
  c.next_eval = s.next_eval;
  c.k1 = 0;
  c.k7 = 6;
  c.fresh = 1;
  c.midstep = s.status == MARLPDE_STATUS_STEP_BUDGET_MIDSTEP ? 1 : 0;
  c.rejected = c.midstep;
  c.ysl = 0;
  c.locate = 0;
  c.ev_prev = 0u;
  c.skip = 0;
  if (s.t >= A.opt.t_bound) {
    c.active = 0;
    c.status = MARLPDE_STATUS_FINISHED;
  }
  A.ctl[col] = c;            // buffer 0: read by the first stage-0 launch and the first prepare
  A.ctl[A.B + col] = c;
}

__global__ void finish_kernel(const Args A, int parity) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= A.B) return;
  const Ctl c = A.ctl[(size_t)parity * A.B + col];
  marlpde_column_state s;
  s.t = c.t;
  s.h_abs = c.h_abs;
  s.n_accepted = c.n_acc;
  s.n_rejected = c.n_rej;
  s.nfev = c.nfev;
  s.status = c.active ? (c.rejected ? MARLPDE_STATUS_STEP_BUDGET_MIDSTEP : MARLPDE_STATUS_STEP_BUDGET) : c.status;
  s.next_eval = c.next_eval;
  A.state[col] = s;
}

struct Cells {               // what a thread knows about its two cells
  int col, pair, cell0;
  bool v0, v1;
  size_t base;               // offset of (col, field 0, cell0) inside a [B][5][N] vector
};

__device__ __forceinline__ Cells my_cells(const Args& A) {
  Cells m;
  m.col = blockIdx.x / A.tiles;
  m.pair = (blockIdx.x - m.col * A.tiles) * kThreads + threadIdx.x;
  m.cell0 = 2 * m.pair;
  m.v0 = m.cell0 < A.N;
  m.v1 = m.cell0 + 1 < A.N;
  m.base = (size_t)m.col * 5 * A.N + m.cell0;
  return m;
}

// y ping-pongs between the caller's array and workspace vector 0 (an accepted step flips the index instead of copying
// y_new over y)
__device__ __forceinline__ double* ybuf(const Args& A, int sl) { return sl ? A.tile : A.y; }

// two adjacent cells of field f from a [B][5][N] vector (N may be odd: no 16-byte loads)
__device__ __forceinline__ void ld2(const double* v, const Cells& m, int f, int N, double& a, double& b) {
  const double* p = v + m.base + (size_t)f * N;
  a = m.v0 ? p[0] : 0.0;
  b = m.v1 ? p[1] : 0.0;
}
__device__ __forceinline__ void st2(double* v, const Cells& m, int f, int N, double a, double b) {
  double* p = v + m.base + (size_t)f * N;
  if (m.v0) p[0] = a;
  if (m.v1) p[1] = b;
}

// end of a call: columns whose y lives in the workspace buffer are copied back to the caller's array
__global__ void __launch_bounds__(kThreads) copyback_kernel(const Args A, int parity) {
  const Cells m = my_cells(A);
  if (A.ctl[(size_t)parity * A.B + m.col].ysl == 0) return;
#pragma unroll
  for (int f = 0; f < 5; ++f) {
    double a, b;
    ld2(A.tile, m, f, A.N, a, b);
    st2(A.y, m, f, A.N, a, b);
  }
}

__device__ __forceinline__ double* partials_of(const Args& A, int parity, int col) {
  return A.partials + ((size_t)parity * A.B + col) * A.pstride;
}
__device__ __forceinline__ unsigned* evpart_of(const Args& A, int parity, int col) {
  return A.evpart + ((size_t)parity * A.B + col) * A.pstride;
}

// ---- event location (ivp.py handle_events -> solve_event_equation: brentq on the dense output of the step), run by
// ONE CTA of the column: the monitor value at y(t + x h) is a min over all cells of the quartic interpolant (K1, K3..K6,
// K7 and y of the step that has just been recomputed with all its stage derivatives stored).  Same arithmetic as
// rk45_persistent.cu::event_partial, so both paths locate the same roots.  All threads of the CTA call this.
__device__ void locate_events(const Args& A, const Ctl& c, int col, unsigned act, const fm::Tables& tb) {
  __shared__ ColumnConsts kc;
  __shared__ double redm[32];
  const int N = A.N, n_thr = (int)blockDim.x, n_warps = (n_thr + 31) >> 5;
  const size_t vec = (size_t)A.B * 5 * N;
  if (threadIdx.x == 0) make_consts(A.params[col], N, kc);
  __syncthreads();
  const size_t cb = (size_t)col * 5 * N;
  const double* const Kp[6] = {A.K + (size_t)c.k1 * vec + cb, A.K + 2 * vec + cb, A.K + 3 * vec + cb,
                               A.K + 4 * vec + cb,           A.K + 5 * vec + cb, A.K + (size_t)c.k7 * vec + cb};
  const double* const yo = ybuf(A, c.ysl) + cb;
  auto interp = [&](int f, int cell, double x) -> double {
    const size_t o = (size_t)f * N + cell;
    double qq[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      double sacc = dp::P[0][j] * Kp[0][o];
      sacc = fma(dp::P[2][j], Kp[1][o], sacc);
      sacc = fma(dp::P[3][j], Kp[2][o], sacc);
      sacc = fma(dp::P[4][j], Kp[3][o], sacc);
      sacc = fma(dp::P[5][j], Kp[4][o], sacc);
      qq[j] = fma(dp::P[6][j], Kp[5][o], sacc);
    }
    const double poly = x * (qq[0] + x * (qq[1] + x * (qq[2] + x * qq[3])));
    return fma(c.h, poly, yo[o]);
  };
  while (act) {
    const int k = __ffs(act) - 1;
    act &= act - 1u;
    BrentState bs;
    bs.init(c.t, c.t_new);
    double xeval = c.t;
    for (;;) {
      const double x = (xeval - c.t) / c.h;
      double v = INFINITY;
      for (int cell = threadIdx.x; cell < N; cell += n_thr) {
        double w;
        if (k == 0) {
          w = fmin(fmin(fmin(interp(0, cell, x), interp(1, cell, x)), fmin(interp(2, cell, x), interp(3, cell, x))),
                   interp(4, cell, x));
        } else if (k == 1) {
          w = interp(0, cell, x);
        } else if (k == 2) {
          w = interp(1, cell, x);
        } else if (k == 3) {
          w = -(interp(0, cell, x) + interp(1, cell, x));
        } else {
          const double Phi = interp(4, cell, x);
          if (k == 4) {
            w = -Phi;
          } else {
            const double F = 1.0 - fm::exp(tb, fma(-10.0, fm::rcp3(Phi), 10.0));
            const double Phi2 = Phi * Phi;
            w = k == 5 ? fma(kc.rhorat * (Phi2 * Phi), F * fm::rcp3(1.0 - Phi), kc.presum)
                       : -fma(-kc.rhorat * Phi2, F, kc.presum);
          }
        }
        v = fmin(v, w);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
      __syncthreads();                                      // the previous round's redm reads are done
      if ((threadIdx.x & 31) == 0) redm[threadIdx.x >> 5] = v;
      __syncthreads();
      double mval = redm[0];
      for (int w = 1; w < n_warps; ++w) mval = fmin(mval, redm[w]);
      const double g = (k == 3 || k == 4) ? (-mval) - 1.0 : (k == 6 ? -mval : mval);
      double root = 0.0;
      if (bs.feed(g, xeval, root)) {                        // (uniform: every thread holds the same state)
        if (threadIdx.x == 0) {
          int32_t* cnt = A.ev_counts + (size_t)col * MARLPDE_NEVENTS + k;
          const int n = *cnt;
          if (n < A.opt.event_capacity)
            A.ev_times[((size_t)col * MARLPDE_NEVENTS + k) * A.opt.event_capacity + n] = root;
          *cnt = n + 1;
        }
        break;
      }
    }
  }
}

// ---- close the previous attempt of a column (error norm -> accept/reject -> new h, dense output, y <- y_new, FSAL slot
// swap) and begin the next one.  Reads control buffer `pin` (and the partial sums / predicate words of parity `pin`),
// publishes the new control block in `pin ^ 1` (first CTA of the column) and returns it: every CTA of a column derives
// the same block from the same inputs.  `m` = the cells this THREAD writes dense-output samples for.  Called by every
// thread of the CTA (the event location inside has block barriers).  `run` = whether the attempt described by the
// returned block is to be run by the caller now (false for a column that is done, and for the launch in which the
// events of a step were located: the locating CTA reads every cell's stage derivatives, so no CTA of the column may
// start overwriting them).
__device__ Ctl close_and_begin(const Args& A, int pin, const Cells& m, bool first_cta, const fm::Tables& tb, bool& run) {
  const int N = A.N;
  const size_t vec = (size_t)A.B * 5 * N;
  Ctl c = A.ctl[(size_t)pin * A.B + m.col];
  const bool publisher = first_cta && threadIdx.x == 0;
  const bool ev_on = (A.opt.flags & MARLPDE_FLAG_EVENTS) != 0;
  run = false;
  if (!c.active) {
    if (publisher) A.ctl[(size_t)(pin ^ 1) * A.B + m.col] = c;
    return c;
  }
  if (c.skip) {                                // committed in the previous launch, not run yet: nothing to close
    c.skip = 0;
    run = true;
    if (publisher) A.ctl[(size_t)(pin ^ 1) * A.B + m.col] = c;
    return c;
  }
  bool located = false;
  const double* const K1 = A.K + (size_t)c.k1 * vec;
  if (!c.fresh) {
    // ---- error norm of the attempt that just ran: per-window partial sums, fixed order
    double sum = 0.0;
    const int n_part = A.tiles2;
    const double* part = partials_of(A, pin, m.col);
    for (int i = 0; i < n_part; ++i) sum += part[i];
    const double err_norm = sqrt(sum / (double)(5 * N));
    c.nfev += 6;
    c.attempts += 1;
    // ---- event monitors (MARLPDE_FLAG_EVENTS): sign classes of the 7 monitors at y_new from the per-window predicate
    // bits the attempt kernel left behind; every CTA of the column derives the same decision
    bool replay = false;
    unsigned ev_new = 0u;
    if (ev_on && err_norm < 1.0) {
      const unsigned* evp = evpart_of(A, pin, m.col);
      for (int i = 0; i < n_part; ++i) ev_new |= evp[i];
      unsigned act = 0u;
      if (ev_new != c.ev_prev || (ev_new & kEqBitsMask) != 0u)
        act = active_events(event_classes(c.ev_prev), event_classes(ev_new));
      if (act) {
        if (c.locate == 0) {
          // first sight: the attempt ran without storing K3..K6.  Do not commit; the next launch repeats the very same
          // attempt (same y, K1, h) with all stage derivatives stored, then the roots are located below.
          c.locate = 1;
          replay = true;
          c.nfev -= 6;
          c.attempts -= 1;
        } else {
          if (first_cta) locate_events(A, c, m.col, act, tb);   // CTA-uniform
          c.locate = 0;
          located = true;
        }
      }
    }
    if (replay) {
      // nothing changes: same step again
    } else if (err_norm < 1.0) {
      if (ev_on) c.ev_prev = ev_new;
      double factor = dp::MAX_FACTOR;
      if (err_norm != 0.0) factor = fmin(dp::MAX_FACTOR, dp::SAFETY * fm::exp(tb, -0.2 * fm::log(tb, err_norm)));
      if (c.rejected) factor = fmin(1.0, factor);
      const double* K7 = A.K + (size_t)c.k7 * vec;
      // dense output for t_eval points in (t, t_new]
      int ne = c.next_eval;
      while (ne < A.opt.n_eval) {
        const double te = A.t_eval[ne];
        if (!(te <= c.t_new)) break;
        const double x = (te - c.t) / c.h;
#pragma unroll 1
        for (int f = 0; f < 5; ++f) {
          double k[6][2], yv[2];
          ld2(K1, m, f, N, k[0][0], k[0][1]);
          ld2(A.K + 2 * vec, m, f, N, k[1][0], k[1][1]);
          ld2(A.K + 3 * vec, m, f, N, k[2][0], k[2][1]);
          ld2(A.K + 4 * vec, m, f, N, k[3][0], k[3][1]);
          ld2(A.K + 5 * vec, m, f, N, k[4][0], k[4][1]);
          ld2(K7, m, f, N, k[5][0], k[5][1]);
          ld2(ybuf(A, c.ysl), m, f, N, yv[0], yv[1]);
          double out[2];
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            double qq[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              double s = dp::P[0][j] * k[0][q];
              s = fma(dp::P[2][j], k[1][q], s);
              s = fma(dp::P[3][j], k[2][q], s);
              s = fma(dp::P[4][j], k[3][q], s);
              s = fma(dp::P[5][j], k[4][q], s);
              qq[j] = fma(dp::P[6][j], k[5][q], s);
            }
            out[q] = fma(c.h, x * (qq[0] + x * (qq[1] + x * (qq[2] + x * qq[3]))), yv[q]);
          }
          double* sp = A.snap + ((size_t)m.col * A.opt.n_eval + ne) * 5 * N + (size_t)f * N + m.cell0;
          if (m.v0) sp[0] = out[0];
          if (m.v1) sp[1] = out[1];
        }
        ++ne;
      }
      c.next_eval = ne;
      // accept: y <- y_new (written to the other y buffer: flip the index), K1 <-> K7
      c.ysl ^= 1;
      const int tmp = c.k1;
      c.k1 = c.k7;
      c.k7 = tmp;
      c.t = c.t_new;
      c.h_abs *= factor;
      c.n_acc += 1;
      if (c.t >= A.opt.t_bound) {
        c.active = 0;
        c.status = MARLPDE_STATUS_FINISHED;
      } else {
        begin_step(c, A.opt);
        if (!begin_attempt(c, A.opt)) {
          c.active = 0;
          c.status = MARLPDE_STATUS_STEP_TOO_SMALL;
        }
      }
    } else {
      c.h_abs *= fmax(dp::MIN_FACTOR, dp::SAFETY * fm::exp(tb, -0.2 * fm::log(tb, err_norm)));
      c.rejected = 1;
      c.n_rej += 1;
      if (!begin_attempt(c, A.opt)) {
        c.active = 0;
        c.status = MARLPDE_STATUS_STEP_TOO_SMALL;
      }
    }
  } else {
    c.fresh = 0;
    if (ev_on) {                               // monitors at the start point (ivp.py: g = event(t0, y0)), from the K1 launch
      const unsigned* evp = evpart_of(A, pin, m.col);       // (written by the K1 launch, parity 0 = the first `pin`)
      unsigned b = 0u;
      for (int i = 0; i < A.tiles; ++i) b |= evp[i];
      c.ev_prev = b;
    }
    if (c.nfev == 0) c.nfev = 1;               // K1 of a resumed column replaces the FSAL value: not counted again
    if (!c.midstep) begin_step(c, A.opt);      // a mid-step resume continues the step it was in
    c.midstep = 0;
    if (!begin_attempt(c, A.opt)) {
      c.active = 0;
      c.status = MARLPDE_STATUS_STEP_TOO_SMALL;
    }
  }
  run = c.active != 0 && !located;
  if (c.active && located) c.skip = 1;                      // the attempt begun here runs in the NEXT launch
  if (publisher) A.ctl[(size_t)(pin ^ 1) * A.B + m.col] = c;
  return c;
}

// ---- prepare: close_and_begin as a kernel of its own, to close the last attempt of a batch (the attempt kernel closes
// every earlier one in its prologue).
__global__ void __launch_bounds__(kThreads) prepare_kernel(const Args A, int pin) {
  __shared__ __align__(16) unsigned char tab_raw[fm::kTableBytes];
  const fm::Tables tb = fm::stage_tables(tab_raw, threadIdx.x, blockDim.x);
  __syncthreads();
  const Cells m = my_cells(A);
  bool run;
  close_and_begin(A, pin, m, blockIdx.x == m.col * A.tiles, tb, run);
}

// ---- K1 = f(y) at the start of a call (columns still active), and the monitor bits at the start point.  256 cells per
// CTA; a thread's own cells and the two halo cells are read from y in HBM.
__global__ void __launch_bounds__(kThreads, 3) k1_kernel(const Args A) {
  __shared__ ColumnConsts kc;
  __shared__ __align__(16) unsigned char tab_raw[fm::kTableBytes];
  const Cells m = my_cells(A);
  const Ctl c = A.ctl[m.col];                               // control buffer 0, as init_kernel left it
  if (!c.active || !c.fresh) return;                        // uniform per CTA
  const fm::Tables tb = fm::stage_tables(tab_raw, threadIdx.x, blockDim.x);
  const int N = A.N;
  if (threadIdx.x == 0) make_consts(A.params[m.col], N, kc);
  const size_t vec = (size_t)A.B * 5 * N;

  double cc[5][2], hm[5], hp[5];
#pragma unroll
  for (int f = 0; f < 5; ++f) {
    const double* p = A.y + m.base + (size_t)f * N;
    cc[f][0] = m.v0 ? p[0] : 0.5;
    cc[f][1] = m.v1 ? p[1] : 0.5;
    hm[f] = (m.v0 && m.cell0 > 0) ? p[-1] : 0.0;
    hp[f] = (m.cell0 + 2 < N) ? p[2] : 0.0;
  }
  __syncthreads();                                          // kc and the tables are staged

  double mlo[5], phi[5];
#pragma unroll
  for (int f = 0; f < 5; ++f) {
    mlo[f] = (m.v0 && m.cell0 > 0) ? hm[f] : top_ghost(kc, f, cc[f][0]);
    if (m.cell0 + 2 < N) {
      phi[f] = hp[f];
    } else if (m.v1) {
      phi[f] = bottom_ghost(f, cc[f][1], cc[f][0]);
    } else {
      cc[f][1] = bottom_ghost(f, cc[f][0], mlo[f]);
      phi[f] = cc[f][1];
    }
  }
  const bool in_mask[2] = {m.cell0 >= kc.mask_lo && m.cell0 < kc.mask_hi,
                           m.cell0 + 1 >= kc.mask_lo && m.cell0 + 1 < kc.mask_hi};
  double r[5][2], U[2], W[2];
  // (kVarDPhi = true: bit-identical for columns without MARLPDE_MODEL_VAR_DPHI; runs once per call)
  PairFlags fl = rhs_pair<rhs_schedule(kSchedSplit), true>(kc, tb, cc, mlo, phi, in_mask, r, U, W);
  fl.bad[0] = fl.bad[0] && m.v0;
  fl.bad[1] = fl.bad[1] && m.v1;
  if (fl.bad[0] || fl.bad[1]) rhs_pair_fixup(kc, tb, fl, cc, mlo, phi, in_mask, r, U, W);

  double* const K1 = A.K + (size_t)c.k1 * vec;
#pragma unroll
  for (int f = 0; f < 5; ++f) st2(K1, m, f, N, r[f][0], r[f][1]);
  if (A.opt.flags & MARLPDE_FLAG_EVENTS) {                 // monitor signs at the start point (U, W come with K1)
    __shared__ unsigned sbits[kThreads / 32];
    const unsigned bw = __reduce_or_sync(0xffffffffu, event_bits_sel(cc, U, W, m.v0, m.v1));
    if ((threadIdx.x & 31) == 0) sbits[threadIdx.x >> 5] = bw;
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned b = 0u;
      for (int w = 0; w < kThreads / 32; ++w) b |= sbits[w];
      evpart_of(A, 0, m.col)[blockIdx.x - m.col * A.tiles] = b;
    }
  }
}


// =================================================================================================
// Overlapped tiles: ONE launch per step attempt.  A 320-thread CTA integrates a 640-cell window of a
// long column through all six stages and the FSAL evaluation ON CHIP, exactly like a slot of the
// persistent kernel (y, K1, stage input and stage derivative in registers, K2..K5 and the halo
// exchange tile in shared memory).  Neighbouring windows overlap by 2 x 6 cells: a stage evaluation
// invalidates one more cell at each window edge (its neighbour lies outside the window), so after
// K2..K7 the inner 628 cells are exact and only those are written back.  HBM traffic per attempt is
// 4 vector passes (read y, K1; write y_new, K7), at 1.9 % redundant arithmetic.
// =================================================================================================
// Window sizes: 320 threads (640-cell windows, 628 owned cells) when the batch fills the machine; 128 threads (256-cell
// windows, 244 owned) for small batches — N = 20 000 x 1 is 32 large windows on 148 SMs, and an attempt cannot be
// faster than one CTA's six stage trips (~5 200 cycles each with 10 warps in lock-step, ~2 500 with one warp per
// scheduler): more, smaller windows cut that latency at 4.9 % instead of 1.9 % redundant arithmetic.
constexpr int kTileHalo = 6;
constexpr int kTileThreadsLarge = 320, kTileThreadsSmall = 128;
__host__ __device__ constexpr int tile_valid_cells(int threads) { return 2 * threads - 2 * kTileHalo; }

template <int TT>
struct TileSmemT {
  static constexpr size_t off_K = 0;                                                   // double2 [4][5][TT]
  static constexpr size_t off_E = off_K + sizeof(double2) * 4 * 5 * TT;                // double [2][5][TT]
  static constexpr size_t off_O = off_E + sizeof(double) * 2 * 5 * TT;
  static constexpr size_t off_tab = off_O + sizeof(double) * 2 * 5 * TT;
  static constexpr size_t off_kc = off_tab + fm::kTableBytes;
  static constexpr size_t off_red = off_kc + (sizeof(ColumnConsts) + 15) / 16 * 16;
  static constexpr size_t off_bar = off_red + 16 * sizeof(double);                      // mbarrier
  static constexpr size_t total = off_bar + 16;
  static_assert(total <= 227 * 1024, "tile kernel shared memory");
};

// VD: batches with MARLPDE_MODEL_VAR_DPHI columns (opt.flags & MARLPDE_FLAG_VAR_DPHI); EV: MARLPDE_FLAG_EVENTS
template <bool VD, bool EV, int TT>
__global__ void __launch_bounds__(TT, 1) tile_attempt_kernel(const Args A, int pin) {
  MARLPDE_DYN_SMEM(smem_raw);
  using TileSmem = TileSmemT<TT>;
  constexpr int kTileThreads = TT, kTileCells = 2 * TT, kTileValid = tile_valid_cells(TT);
  constexpr int TP = kTileThreads;
  const int tid = threadIdx.x;
  const int col = blockIdx.x / A.tiles2;
  const int tile = blockIdx.x - col * A.tiles2;
  const int N = A.N;
  const fm::Tables tb = fm::stage_tables(smem_raw + TileSmem::off_tab, tid, blockDim.x);
  __syncthreads();
  // ---- prologue (r02q): close the PREVIOUS attempt of the column and begin this one — what used to be a launch of
  // its own (prepare_kernel) between two attempts.  Every CTA of the column derives the same control block; this thread
  // writes the dense-output samples of the cells its window owns.  One launch per attempt instead of two: a batch of a
  // few columns is bound by launch latency (N = 20 000 x 1: 49.8 k -> see DESIGN.md section 9, r02q).
  Ctl c0;
  {
    const int pe0 = 2 * tid, pg0 = tile * kTileValid - kTileHalo + pe0;
    Cells mt;
    mt.col = col;
    mt.pair = 0;
    mt.cell0 = pg0 < 0 ? 0 : pg0;
    mt.v0 = pg0 >= 0 && pg0 < N && pe0 >= kTileHalo && pe0 < kTileCells - kTileHalo;
    mt.v1 = pg0 + 1 >= 0 && pg0 + 1 < N && pe0 + 1 >= kTileHalo && pe0 + 1 < kTileCells - kTileHalo;
    mt.base = (size_t)col * 5 * N + (size_t)mt.cell0;
    bool run;
    c0 = close_and_begin(A, pin, mt, tile == 0, tb, run);
    if (!run) return;                                       // uniform per CTA
  }
  double2* const sK = reinterpret_cast<double2*>(smem_raw + TileSmem::off_K) + tid;
  double* const sE = reinterpret_cast<double*>(smem_raw + TileSmem::off_E);
  double* const sO = reinterpret_cast<double*>(smem_raw + TileSmem::off_O);
  ColumnConsts& kc = *reinterpret_cast<ColumnConsts*>(smem_raw + TileSmem::off_kc);
  double* const red = reinterpret_cast<double*>(smem_raw + TileSmem::off_red);
  uint64_t* const sBar = reinterpret_cast<uint64_t*>(smem_raw + TileSmem::off_bar);   // split barrier of the stage loop
  if (tid == 0) mbar_init(sBar, blockDim.x);
  unsigned bar_parity = 0;
  if (tid == 0) make_consts(A.params[col], N, kc);
  const size_t vec = (size_t)A.B * 5 * N;
  const double h = c0.h;

  const int e0 = 2 * tid;                                   // position inside the window
  const int g0 = tile * kTileValid - kTileHalo + e0;        // global cell of my first cell (always even)
  const bool in0 = g0 >= 0 && g0 < N, in1 = g0 + 1 >= 0 && g0 + 1 < N;
  const bool top = g0 == 0;                                 // my first cell is the column's first cell
  const bool bot1 = g0 + 1 == N - 1;                        // my second cell is the column's last cell
  const bool bot0 = g0 == N - 1;                            // odd N: my first cell is the last one
  const bool out0 = in0 && e0 >= kTileHalo && e0 < kTileCells - kTileHalo;      // cells this window owns
  const bool out1 = in1 && e0 + 1 >= kTileHalo && e0 + 1 < kTileCells - kTileHalo;
  const size_t base = (size_t)col * 5 * N + (size_t)(g0 < 0 ? 0 : g0);
  const double* const haloM = sO + (tid == 0 ? tid : tid - 1);
  const double* const haloP = sE + (tid == TP - 1 ? tid : tid + 1);
  double* const myE = sE + tid;
  double* const myO = sO + tid;
  auto Kslot = [&](int logical) -> double* {
    const int s = logical == 1 ? c0.k1 : (logical == 7 ? c0.k7 : logical - 1);
    return A.K + (size_t)s * vec;
  };
  auto Kst = [&](int s, int f, double v0, double v1) { sK[(s * 5 + f) * TP] = make_double2(v0, v1); };
  auto Kld = [&](int s, int f) -> double2 { return sK[(s * 5 + f) * TP]; };

  double y[5][2], k1[5][2], c[5][2], r[5][2];
  {
    const double* K1g = Kslot(1);
#pragma unroll
    for (int f = 0; f < 5; ++f) {
      const double* yp = ybuf(A, c0.ysl) + base + (size_t)f * N;
      const double* kp = K1g + base + (size_t)f * N;
      y[f][0] = in0 ? yp[0] : 0.5;
      y[f][1] = in1 ? yp[g0 < 0 ? g0 + 1 : 1] : 0.5;     // (g0 = -2k < 0 never has an in-range partner; kept safe)
      k1[f][0] = in0 ? kp[0] : 0.0;
      k1[f][1] = in1 ? kp[g0 < 0 ? g0 + 1 : 1] : 0.0;
    }
  }
  const bool in_mask[2] = {in0 && g0 >= A.params[col].mask_lo && g0 < A.params[col].mask_hi,
                           in1 && g0 + 1 >= A.params[col].mask_lo && g0 + 1 < A.params[col].mask_hi};
  auto tile_store = [&](int b) {
#pragma unroll
    for (int f = 0; f < 5; ++f) {
      myE[(b * 5 + f) * TP] = c[f][0];
      myO[(b * 5 + f) * TP] = c[f][1];
    }
  };
  {
    const double ha = h * dp::a21;
#pragma unroll
    for (int f = 0; f < 5; ++f) {
      c[f][0] = fma(ha, k1[f][0], y[f][0]);
      c[f][1] = fma(ha, k1[f][1], y[f][1]);
    }
    tile_store(1);
  }
  __syncthreads();

  double U[2], W[2];
#pragma unroll 1
  for (int i = 1; i <= 6; ++i) {
    // the neighbour-free part of the RHS overlaps the pending barrier (see rk45_persistent.cu)
    OwnTerms own;
    PairFlags fl = rhs_pair_own<rhs_schedule(kSchedLean), VD>(kc, tb, c, in_mask, own);
    if (i > 1) {
      mbar_wait(sBar, bar_parity);
      bar_parity ^= 1u;
    }
    const int tb_ = (i & 1) * 5 * TP;
    double mlo[5], phi[5];
#pragma unroll
    for (int f = 0; f < 5; ++f) {
      const double hm = haloM[tb_ + f * TP], hp = haloP[tb_ + f * TP];
      mlo[f] = top ? top_ghost(kc, f, c[f][0]) : (tid == 0 ? c[f][0] : hm);
      if (bot1) {
        phi[f] = bottom_ghost(f, c[f][1], c[f][0]);
      } else if (bot0) {
        c[f][1] = bottom_ghost(f, c[f][0], mlo[f]);
        phi[f] = c[f][1];
      } else {
        phi[f] = tid == TP - 1 ? c[f][1] : hp;
      }
    }
    rhs_pair_finish<VD>(kc, c, mlo, phi, own, r);
    U[0] = own.U[0];
    U[1] = own.U[1];
    W[0] = own.W[0];
    W[1] = own.W[1];
    // cells a stage can still compute correctly: i window cells are lost at either edge by stage i
    fl.bad[0] = fl.bad[0] && in0 && e0 >= i && e0 < kTileCells - i;
    fl.bad[1] = fl.bad[1] && in1 && e0 + 1 >= i && e0 + 1 < kTileCells - i;
    if (fl.bad[0] || fl.bad[1]) rhs_pair_fixup(kc, tb, fl, c, mlo, phi, in_mask, r, U, W);
#pragma unroll
    for (int f = 0; f < 5; ++f) {                            // cells outside the column stay inert
      if (!in0) r[f][0] = 0.0;
      if (!in1) r[f][1] = 0.0;
    }
    switch (i) {
      case 1:
#pragma unroll
        for (int f = 0; f < 5; ++f) {
          Kst(0, f, r[f][0], r[f][1]);
          c[f][0] = fma(h, fma(dp::a31, k1[f][0], dp::a32 * r[f][0]), y[f][0]);
          c[f][1] = fma(h, fma(dp::a31, k1[f][1], dp::a32 * r[f][1]), y[f][1]);
        }
        tile_store(0);
        break;
      case 2:
#pragma unroll
        for (int f = 0; f < 5; ++f) {
          Kst(1, f, r[f][0], r[f][1]);
          const double2 K2 = Kld(0, f);
          c[f][0] = fma(h, fma(dp::a41, k1[f][0], fma(dp::a42, K2.x, dp::a43 * r[f][0])), y[f][0]);
          c[f][1] = fma(h, fma(dp::a41, k1[f][1], fma(dp::a42, K2.y, dp::a43 * r[f][1])), y[f][1]);
        }
        tile_store(1);
        break;
      case 3:
#pragma unroll
        for (int f = 0; f < 5; ++f) {
          Kst(2, f, r[f][0], r[f][1]);
          const double2 K2 = Kld(0, f), K3 = Kld(1, f);
          c[f][0] = fma(h, fma(dp::a51, k1[f][0], fma(dp::a52, K2.x, fma(dp::a53, K3.x, dp::a54 * r[f][0]))), y[f][0]);
          c[f][1] = fma(h, fma(dp::a51, k1[f][1], fma(dp::a52, K2.y, fma(dp::a53, K3.y, dp::a54 * r[f][1]))), y[f][1]);
        }
        tile_store(0);
        break;
      case 4:
#pragma unroll
        for (int f = 0; f < 5; ++f) {
          Kst(3, f, r[f][0], r[f][1]);
          const double2 K2 = Kld(0, f), K3 = Kld(1, f), K4 = Kld(2, f);
          c[f][0] = fma(h, fma(dp::a61, k1[f][0], fma(dp::a62, K2.x, fma(dp::a63, K3.x, fma(dp::a64, K4.x, dp::a65 * r[f][0])))), y[f][0]);
          c[f][1] = fma(h, fma(dp::a61, k1[f][1], fma(dp::a62, K2.y, fma(dp::a63, K3.y, fma(dp::a64, K4.y, dp::a65 * r[f][1])))), y[f][1]);
        }
        tile_store(1);
        break;
      case 5:
#pragma unroll
        for (int f = 0; f < 5; ++f) {
          const double2 K3 = Kld(1, f), K4 = Kld(2, f), K5 = Kld(3, f);
          Kst(0, f, r[f][0], r[f][1]);                       // K6 over the dead K2
          c[f][0] = fma(h, fma(dp::b1, k1[f][0], fma(dp::b3, K3.x, fma(dp::b4, K4.x, fma(dp::b5, K5.x, dp::b6 * r[f][0])))), y[f][0]);
          c[f][1] = fma(h, fma(dp::b1, k1[f][1], fma(dp::b3, K3.y, fma(dp::b4, K4.y, fma(dp::b5, K5.y, dp::b6 * r[f][1])))), y[f][1]);
        }
        tile_store(0);
        break;
      default:
        break;
    }
    if (i < 6) mbar_arrive(sBar);
  }
  // ---- r = K7 = f(y_new), c = y_new: error contribution of the cells this window owns, write-back
  // K3..K6 go to HBM only when the dense output will be needed: a t_eval sample inside the step, or the replay of a
  // step whose events are about to be located
  const bool sample = (c0.next_eval < A.opt.n_eval && A.t_eval[c0.next_eval] <= c0.t_new) || (EV && c0.locate != 0);
  double part = 0.0;
  double* const ynew = ybuf(A, c0.ysl ^ 1);                  // the y buffer that is not in use
  double* const K7g = Kslot(7);
#pragma unroll
  for (int f = 0; f < 5; ++f) {
    const double2 K3 = Kld(1, f), K4 = Kld(2, f), K5 = Kld(3, f), K6 = Kld(0, f);
    const double e0v = fma(dp::e1, k1[f][0], fma(dp::e3, K3.x, fma(dp::e4, K4.x, fma(dp::e5, K5.x, fma(dp::e6, K6.x, dp::e7 * r[f][0])))));
    const double e1v = fma(dp::e1, k1[f][1], fma(dp::e3, K3.y, fma(dp::e4, K4.y, fma(dp::e5, K5.y, fma(dp::e6, K6.y, dp::e7 * r[f][1])))));
    const double s0 = fma(fmax(fabs(y[f][0]), fabs(c[f][0])), A.opt.rtol, A.opt.atol);
    const double s1 = fma(fmax(fabs(y[f][1]), fabs(c[f][1])), A.opt.rtol, A.opt.atol);
    const double z0 = (h * e0v) * fm::rcp3(s0), z1 = (h * e1v) * fm::rcp3(s1);
    if (out0) part = fma(z0, z0, part);
    if (out1) part = fma(z1, z1, part);
    const size_t o = base + (size_t)f * N;
    if (out0) {
      ynew[o] = c[f][0];
      K7g[o] = r[f][0];
    }
    if (out1) {
      ynew[o + 1] = c[f][1];
      K7g[o + 1] = r[f][1];
    }
    if (sample) {                                            // K3..K6 are only needed by the dense output
      if (out0) {
        A.K[2 * vec + o] = K3.x;
        A.K[3 * vec + o] = K4.x;
        A.K[4 * vec + o] = K5.x;
        A.K[5 * vec + o] = K6.x;
      }
      if (out1) {
        A.K[2 * vec + o + 1] = K3.y;
        A.K[3 * vec + o + 1] = K4.y;
        A.K[4 * vec + o + 1] = K5.y;
        A.K[5 * vec + o + 1] = K6.y;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((tid & 31) == 0) red[tid >> 5] = part;
  if constexpr (EV) {     // predicate bits of the monitors at y_new over the cells this window owns (U, W come with K7)
    const unsigned bw = __reduce_or_sync(0xffffffffu, event_bits_sel(c, U, W, out0, out1));
    if ((tid & 31) == 0) reinterpret_cast<unsigned*>(red + kTileThreads / 32)[tid >> 5] = bw;
  }
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
    for (int w = 0; w < kTileThreads / 32; ++w) s += red[w];
    partials_of(A, pin ^ 1, col)[tile] = s;               // (parity of the control block this attempt ran under)
    if constexpr (EV) {
      unsigned b = 0u;
      for (int w = 0; w < kTileThreads / 32; ++w) b |= reinterpret_cast<unsigned*>(red + kTileThreads / 32)[w];
      evpart_of(A, pin ^ 1, col)[tile] = b;
    }
  }
}

}  // namespace st

size_t rk45_stream_workspace_bytes(int n_columns, int n_cells) { return st::layout(n_columns, n_cells).total; }

namespace {
struct GraphKey {             // everything a captured batch depends on (compared bytewise)
  st::Args a;
  long long attempts;
  int device, small_tiles;
};
}  // namespace

// the tile kernel instantiations: model variant x events x window size
template <bool VD, bool EV, int TT>
static cudaError_t tile_launch(const st::Args& a, unsigned tgrid, int cbuf, cudaStream_t s_) {
#ifndef MARLPDE_HOST_EMU
  static bool configured = false;               // (per instantiation; the attribute is sticky per device context)
  static int configured_device = -1;
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured || configured_device != dev) {
    cudaError_t e = cudaFuncSetAttribute(st::tile_attempt_kernel<VD, EV, TT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)st::TileSmemT<TT>::total);
    if (e != cudaSuccess) return e;
    configured = true;
    configured_device = dev;
  }
#endif
  MARLPDE_LAUNCH((st::tile_attempt_kernel<VD, EV, TT>), tgrid, TT, (st::TileSmemT<TT>::total), s_, a, cbuf);
  return cudaSuccess;
}

template <int TT>
static cudaError_t tile_dispatch(bool vd, bool ev, const st::Args& a, unsigned tgrid, int cbuf, cudaStream_t s_) {
  if (vd && ev) return tile_launch<true, true, TT>(a, tgrid, cbuf, s_);
  if (vd) return tile_launch<true, false, TT>(a, tgrid, cbuf, s_);
  if (ev) return tile_launch<false, true, TT>(a, tgrid, cbuf, s_);
  return tile_launch<false, false, TT>(a, tgrid, cbuf, s_);
}

cudaError_t launch_rk45_stream(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                               int n_columns, int n_cells, const marlpde_rk45_options& opt, const double* d_t_eval,
                               double* d_snap, int32_t* d_ev_counts, double* d_ev_times, void* d_work,
                               long long attempts, cudaStream_t stream) {
  const st::Layout L = st::layout(n_columns, n_cells);
  unsigned char* w = static_cast<unsigned char*>(d_work);
  st::Args a;
  std::memset(&a, 0, sizeof a);               // (padding bytes take part in the graph-cache comparison)
  a.y = d_y;
  a.params = d_params;
  a.state = d_state;
  a.t_eval = d_t_eval;
  a.snap = d_snap;
  a.K = reinterpret_cast<double*>(w + L.off_K);
  a.tile = reinterpret_cast<double*>(w + L.off_tile);
  a.partials = reinterpret_cast<double*>(w + L.off_part);
  a.ctl = reinterpret_cast<st::Ctl*>(w + L.off_ctl);
  a.evpart = reinterpret_cast<unsigned*>(w + L.off_ev);
  a.ev_counts = d_ev_counts;
  a.ev_times = d_ev_times;
  a.B = n_columns;
  a.N = n_cells;
  a.tiles = (n_cells + st::kCellsPerCta - 1) / st::kCellsPerCta;
  a.pstride = (n_cells + 243) / 244 + 1;
  a.opt = opt;
  const long long blocks = (long long)a.tiles * n_columns;
  if (blocks > 0x7fffffffLL) return cudaErrorInvalidValue;
  const unsigned grid = (unsigned)blocks;
  const unsigned cgrid = (unsigned)((n_columns + 127) / 128);
  // window size (MARLPDE_RK45_TILE=small|large overrides)
  int sms = 148, dev = 0;
#ifndef MARLPDE_HOST_EMU
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
#endif
  (void)dev;
  const int valid_l = st::tile_valid_cells(st::kTileThreadsLarge), valid_s = st::tile_valid_cells(st::kTileThreadsSmall);
  // small windows while ALL of them are resident at once (two 128-thread CTAs per SM: one wave at about two thirds
  // of a large window's latency).  Measured (r02f, r02l; column-steps/s, small vs large): 20 000 x 1 49.6 k / 41.5 k,
  // 20 000 x 3 130 k / 121 k, 5 000 x 12 567 k / 504 k, 2 000 x 32 1.53 M / 1.36 M — but 20 000 x 4 (328 small CTAs:
  // two waves) 127 k / 160 k and 20 000 x 8 162 k / 176 k.
  const long long ctas_small = (long long)((n_cells + valid_s - 1) / valid_s) * n_columns;
  bool small_tiles = ctas_small <= 2LL * sms;
  const char* tile_env = std::getenv("MARLPDE_RK45_TILE");
  if (tile_env && tile_env[0] == 's') small_tiles = true;
  if (tile_env && tile_env[0] == 'l') small_tiles = false;
  const int valid = small_tiles ? valid_s : valid_l;
  a.tiles2 = (n_cells + valid - 1) / valid;
  const unsigned tgrid = (unsigned)((long long)a.tiles2 * n_columns);
  const bool var_dphi = (opt.flags & MARLPDE_FLAG_VAR_DPHI) != 0;
  const bool ev_on = (opt.flags & MARLPDE_FLAG_EVENTS) != 0;
  auto enqueue = [&](cudaStream_t s_) -> cudaError_t {
    MARLPDE_LAUNCH(st::init_kernel, cgrid, 128, 0, s_, a);
    MARLPDE_LAUNCH(st::k1_kernel, grid, st::kThreads, 0, s_, a);
    int pin = 0;
    // the tile kernel closes the previous attempt in its prologue: ONE launch per attempt; the prepare launch after the
    // loop only closes the last attempt
    for (long long j = 0; j < attempts; ++j) {
      const cudaError_t et = small_tiles ? tile_dispatch<st::kTileThreadsSmall>(var_dphi, ev_on, a, tgrid, pin, s_)
                                         : tile_dispatch<st::kTileThreadsLarge>(var_dphi, ev_on, a, tgrid, pin, s_);
      if (et != cudaSuccess) return et;
      pin ^= 1;
    }
    MARLPDE_LAUNCH(st::prepare_kernel, grid, st::kThreads, 0, s_, a, pin);
    pin ^= 1;
    MARLPDE_LAUNCH(st::copyback_kernel, grid, st::kThreads, 0, s_, a, pin);
    MARLPDE_LAUNCH(st::finish_kernel, cgrid, 128, 0, s_, a, pin);
    return cudaGetLastError();
  };
#ifndef MARLPDE_HOST_EMU
  // The launches of a batch are captured once into a CUDA graph and replayed — a batch of a few columns is bound by launch
  // latency, and the host drivers repeat identical batches (all step state lives in device memory, the kernel arguments
  // do not change).  Measured (r02a, profiles/r02a_ab_candidates.log): N = 20 000 x 1 37.3 -> 42.0 k attempts/s,
  // N = 2 000 x 8 299 -> 353 k, N = 20 000 x 64 234.5 -> 238.3 k.
  if (attempts <= 1024) {
    static std::mutex mu;
    static struct { bool valid; GraphKey key; cudaGraphExec_t exec; cudaStream_t cap; } cache = {false, {}, nullptr, nullptr};
    std::lock_guard<std::mutex> lock(mu);
    GraphKey key;
    std::memset(&key, 0, sizeof key);
    key.a = a;
    key.attempts = attempts;
    key.small_tiles = small_tiles;
    cudaError_t e = cudaGetDevice(&key.device);
    if (e != cudaSuccess) return e;
    if (!(cache.valid && std::memcmp(&cache.key, &key, sizeof key) == 0)) {
      if (cache.exec) cudaGraphExecDestroy(cache.exec);
      if (cache.cap) cudaStreamDestroy(cache.cap);           // (a stream belongs to the device it was created on)
      cache.valid = false;
      cache.exec = nullptr;
      cache.cap = nullptr;
      if ((e = cudaStreamCreateWithFlags(&cache.cap, cudaStreamNonBlocking)) != cudaSuccess) return e;
      if ((e = cudaStreamBeginCapture(cache.cap, cudaStreamCaptureModeThreadLocal)) != cudaSuccess) return e;
      const cudaError_t el = enqueue(cache.cap);
      cudaGraph_t graph = nullptr;
      e = cudaStreamEndCapture(cache.cap, &graph);
      if (el != cudaSuccess || e != cudaSuccess) {
        if (graph) cudaGraphDestroy(graph);
        return el != cudaSuccess ? el : e;
      }
      e = cudaGraphInstantiate(&cache.exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) return e;
      cache.key = key;
      cache.valid = true;
    }
    return cudaGraphLaunch(cache.exec, stream);
  }
#endif
  return enqueue(stream);
}

}  // namespace marlpde
