/*
 * marlpde_b200.h — C ABI of the B200-native integrator for L'Heureux's five coupled
 * diagenetic equations (aragonite CA, calcite CC, pore-water cCa and cCO3, porosity Phi).
 *
 * This is the drop-in boundary for the ONE hot path of
 * astro-turing/Integrating-diagenetic-equations-using-Python ("the reference"):
 *
 *   reference interface                                   replaced by
 *   ---------------------------------------------------   ---------------------------------
 *   LMAHeureuxPorosityDiff.fun_numba / pde_rhs            marlpde_rhs_batch[_dev]
 *     (marlpde/LHeureux_model.py:290-359, :361-522)
 *   LMAHeureuxPorosityDiff.fun (NumPy backend, :162-288)  marlpde_rhs_batch[_dev] (same maths)
 *   scipy.integrate.solve_ivp(method="RK45", ...)         marlpde_rk45_integrate[_dev]
 *     call site marlpde/Evolve_scenario.py:104-109
 *   scipy.integrate.solve_ivp(method="Radau", jac_sparsity=jacobian_sparsity())   marlpde_radau_integrate[_dev]
 *     the reference's default Solver (marlpde/parameters.py:150-199, :213)
 *   scipy.integrate.solve_ivp(method="BDF" | "LSODA")    marlpde_bdf_integrate[_dev]
 *   scipy.integrate.solve_ivp(method="RK23" | "DOP853")  marlpde_rk23_integrate[_dev], marlpde_dop853_integrate[_dev]
 *   7 event monitors (LHeureux_model.py:524-593)          event outputs of marlpde_rk45_integrate*
 *   derived constants of __init__ (:31-72, :130-133)      marlpde_column_params (filled by the host
 *                                                          mirror, one struct per sediment column)
 *
 * Conventions
 *   - plain C: pointers + sizes, no C++/torch types. `*_dev` entry points take DEVICE pointers
 *     and a cudaStream_t passed as void* (0 = default stream) and never allocate or synchronise;
 *     the un-suffixed entry points take HOST pointers, pick `device`, do their own
 *     H2D/D2H copies and synchronise before returning.
 *   - state layout: y[column][field][cell], fields in the reference's order
 *     CA, CC, cCa, cCO3, Phi (Evolve_scenario.py:64-65), float64, C-contiguous.
 *   - every function returns MARLPDE_OK (0) or a negative MARLPDE_E* code;
 *     marlpde_last_error() returns a thread-local human readable message.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails
 *     with MARLPDE_ENODEVICE.
 */
#ifndef MARLPDE_B200_H
#define MARLPDE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MARLPDE_ABI_VERSION 2
#define MARLPDE_NFIELDS 5
#define MARLPDE_NEVENTS 7

/* return codes */
#define MARLPDE_OK 0
#define MARLPDE_EINVAL (-1)     /* bad argument */
#define MARLPDE_ENODEVICE (-2)  /* no usable CUDA device */
#define MARLPDE_ECUDA (-3)      /* CUDA runtime error (see marlpde_last_error) */
#define MARLPDE_EUNSUPPORTED (-4) /* shape not supported by this build (e.g. n_cells too large) */

/* per-column integration status, mirrors solve_ivp's sol.status (scipy/integrate/_ivp/ivp.py) */
#define MARLPDE_STATUS_FINISHED 0       /* reached t_bound                                  */
#define MARLPDE_STATUS_STEP_TOO_SMALL (-1) /* "Required step size is less than spacing between numbers." */
#define MARLPDE_STATUS_NONFINITE (-2)   /* state became non-finite and the step size collapsed */
#define MARLPDE_STATUS_STEP_BUDGET 1    /* max_steps attempts used up; (t, h_abs, y) are resumable */
#define MARLPDE_STATUS_STEP_BUDGET_MIDSTEP 2 /* streaming path only: the budget ended inside a step whose last
                                          attempt was rejected; resumable like 1 (pass the state back unchanged:
                                          the next attempt then keeps SciPy's "no growth after a rejection" rule,
                                          so a run cut into batches is bit-identical to an uninterrupted one) */

/*
 * Per-column constants: exactly the scalars the reference passes into pde_rhs
 * (LHeureux_model.py:346-359) after deriving them in __init__ (:31-72, :87-88, :130-133),
 * plus the Dirichlet values of the top boundary (:26-30) and the grid spacing of
 * CartesianGrid([[0, max_depth/Xstar]], [N]) (Evolve_scenario.py:40).
 * The two Heaviside masks (Evolve_scenario.py:51-54) are an interval of cells:
 * not_too_deep*not_too_shallow == 1 on [mask_lo, mask_hi), 0 elsewhere.
 */
typedef struct marlpde_column_params {
  double bc_top[MARLPDE_NFIELDS]; /* CA0, CC0, cCa0, cCO30, Phi0 */
  double dx;          /* (max_depth/Xstar)/N                         */
  double inv_dx;      /* 1/dx                                        */
  double inv_dx2;     /* dx**-2                                      */
  double delta_x;     /* x[1]-x[0] of the cell centres (:23-24)      */
  double presum, rhorat, Da, lambda_;
  double dCa, dCO3, delta, KRat;
  double nu1, nu2, m1, m2, n1, n2;
  double dPhi_fixed, Peclet_min, Peclet_max;
  int32_t FV_switch;
  int32_t mask_lo, mask_hi;
  int32_t model_flags; /* MARLPDE_MODEL_*: model variants the reference toggles by editing its source        */
  double auxcon;      /* beta / (D0Ca b g rhow (PhiNR - PhiInfty)) (:65-66); read only with MARLPDE_MODEL_VAR_DPHI */
} marlpde_column_params;

/* model_flags bit 0: time-varying porosity diffusion coefficient dPhi = auxcon F Phi^3 / (1 - Phi) per cell — the line
 * the reference keeps commented out at LHeureux_model.py:222-223 and :430-431 — instead of dPhi_fixed.  It enters the
 * porosity Peclet number (:239, :452) and dPhi * laplace(Phi) (:285, :519).  Integrations of batches that contain such
 * columns must also set MARLPDE_FLAG_VAR_DPHI in marlpde_rk45_options.flags (it selects the kernel build; without it
 * the per-column flag is ignored).  marlpde_rhs_batch* looks at the per-column flag by itself. */
#define MARLPDE_MODEL_VAR_DPHI 1

/* Options of one batched integration (scipy RK45 / Radau semantics; both steppers take this struct). */
typedef struct marlpde_rk45_options {
  double t_bound;      /* end time (t_span[1]); direction is forward only              */
  double rtol, atol;   /* scale = atol + rtol*max(|y|,|y_new|)                         */
  double max_step;     /* +inf for none                                                */
  int64_t max_steps;   /* step-attempt budget per column per call (<=0: unlimited)     */
  int32_t n_eval;      /* number of t_eval points (may be 0)                           */
  int32_t event_capacity; /* slots per (column,event) in event_times (may be 0)       */
  int32_t flags;       /* MARLPDE_FLAG_*                                               */
  int32_t quantum;     /* on-chip RK45 only, with MARLPDE_FLAG_QUEUE_LOCKS and max_steps > 0: step attempts per
                          work item; 0 = chosen by the library, < 0 = one item per column (no quanta)        */
} marlpde_rk45_options;

#define MARLPDE_FLAG_EVENTS 1u   /* monitor the 7 events and locate their roots */
#define MARLPDE_FLAG_QUEUE_LOCKS 2u /* d_queue holds 1 + 2 n_columns zeroed int32 (work counter, one lock word and one
                                    attempt counter per column): the on-chip RK45 kernel may then cut every column's step budget into
                                    quanta claimed quantum-major, which shortens the partly filled last round of a
                                    launch (results are unchanged: a resumed column is bit-identical)          */
#define MARLPDE_FLAG_QUEUE_TAIL 8u /* with MARLPDE_FLAG_QUEUE_LOCKS and max_steps > 0: only the last columns of the batch (2 x the
                                    resident slots) are cut into quanta, the others are claimed whole — for sweeps whose
                                    columns need different numbers of attempts, ordered longest first (launches without
                                    a step budget do this by themselves)                                              */
#define MARLPDE_FLAG_JAC_FD 16u /* implicit integrators: diagonal 5x5 Jacobian blocks from 5 finite-difference evaluations with
                                 * num_jac's step rule (what SciPy forms) instead of the default — every block analytic in one
                                 * pass, and only for cells ON a switching surface of the model the one-sided difference */
#define MARLPDE_FLAG_VAR_DPHI 4u /* some columns of the batch carry MARLPDE_MODEL_VAR_DPHI (see marlpde_column_params) */

/* Per-column integrator state: input (start/resume point) and output (end point). */
typedef struct marlpde_column_state {
  double t;            /* in: start time;  out: time reached                          */
  double h_abs;        /* in: first_step (or the h_abs to resume with); out: next h   */
  int64_t n_accepted;  /* counters are accumulated across resumed calls               */
  int64_t n_rejected;
  int64_t nfev;
  int32_t status;      /* out: MARLPDE_STATUS_*                                        */
  int32_t next_eval;   /* in/out: index of the next t_eval point to be sampled         */
} marlpde_column_state;

typedef struct marlpde_device_info {
  char name[128];
  int32_t sm_count;
  int32_t cc_major, cc_minor;
  int32_t max_smem_per_block; /* opt-in bytes */
  int64_t total_mem;
} marlpde_device_info;

int marlpde_abi_version(void);
/* sizeof() of the ABI structs as compiled into the library, for binding self-checks:
 * which = 0 marlpde_column_params, 1 marlpde_rk45_options, 2 marlpde_column_state,
 * 3 marlpde_device_info; anything else returns -1. */
int marlpde_struct_size(int which);
const char* marlpde_last_error(void);
int marlpde_device_count(void);
int marlpde_get_device_info(int device, marlpde_device_info* info);

/* The host-pointer entry points take their device scratch from one stream-ordered memory pool per device that keeps at
 * most 256 MB cached between calls (cudaMalloc/cudaFree are slow); this trims the pools to zero. Returns the number of
 * pools trimmed. */
int marlpde_release_cached_memory(void);

/* Largest n_cells the on-chip (shared-memory resident) RK45 kernel accepts, and the
 * number of columns one CTA integrates side by side for a given n_cells. */
int marlpde_rk45_max_cells(void);
int marlpde_rk45_columns_per_cta(int n_cells);

/* ---- single RHS call for a batch of columns (replaces fun_numba/pde_rhs) -------------- */
int marlpde_rhs_batch_dev(const double* d_y, const marlpde_column_params* d_params,
                          int n_columns, int n_cells, double* d_out, void* stream);
int marlpde_rhs_batch(const double* y, const marlpde_column_params* params,
                      int n_columns, int n_cells, double* out, int device);

/* ---- batched adaptive RK45 (replaces solve_ivp(method="RK45") per column) ---------------
 *  d_y        [n_columns][5][n_cells]   in: state at state[c].t;  out: state at the time reached
 *  d_state    [n_columns]               in/out, see marlpde_column_state
 *  d_t_eval   [n_eval]                  increasing sample times within [t0, t_bound] (may be NULL)
 *  d_snapshots[n_columns][n_eval][5][n_cells]  dense-output samples (quartic interpolant, as
 *                                       scipy RkDenseOutput); rows >= state.next_eval are untouched
 *  d_event_counts[n_columns][7]         number of roots found per monitor (accumulated)
 *  d_event_times [n_columns][7][event_capacity]  root times (first event_capacity kept)
 *  d_queue    int32 work counter, must be 0 on entry (the kernel claims columns from it); with
 *             MARLPDE_FLAG_QUEUE_LOCKS: 1 + 2 n_columns int32, all 0 on entry
 */
int marlpde_rk45_integrate_dev(double* d_y, const marlpde_column_params* d_params,
                               marlpde_column_state* d_state, int n_columns, int n_cells,
                               const marlpde_rk45_options* opts, const double* d_t_eval,
                               double* d_snapshots, int32_t* d_event_counts,
                               double* d_event_times, int32_t* d_queue, void* stream);
int marlpde_rk45_integrate(double* y, const marlpde_column_params* params,
                           marlpde_column_state* state, int n_columns, int n_cells,
                           const marlpde_rk45_options* opts, const double* t_eval,
                           double* snapshots, int32_t* event_counts, double* event_times,
                           int device);
/* Stream-ordered variant of the host-pointer call, for sweep drivers that overlap the copies of one batch with the
 * kernel of another: H2D copies (one cudaMemcpyAsync per buffer), the launch, the D2H copies and the release of the
 * device scratch are all enqueued on `stream` (a cudaStream_t) and the call returns WITHOUT synchronising.  The host
 * buffers must be page-locked for the copies to be asynchronous and must stay valid and untouched until the caller has
 * synchronised the stream.  Depth grids outside the on-chip range (streaming path) are served synchronously. */
int marlpde_rk45_integrate_async(double* y, const marlpde_column_params* params,
                                 marlpde_column_state* state, int n_columns, int n_cells,
                                 const marlpde_rk45_options* opts, const double* t_eval,
                                 double* snapshots, int32_t* event_counts, double* event_times,
                                 int device, void* stream);

/* ---- the same RK45 for depth grids that do not fit on chip (n_cells up to millions): overlapped 640-cell windows
 * integrated on chip, one launch per step attempt, state and K1 / K7 streaming through HBM (csrc/rk45_streaming.cu).
 *  Arguments as for marlpde_rk45_integrate_dev (marlpde_rk45_stream_integrate_events_dev takes the event outputs and
 *  monitors the 7 events when MARLPDE_FLAG_EVENTS is set; the variant without them rejects the flag), plus
 *  d_workspace  marlpde_rk45_stream_workspace_bytes(n_columns, n_cells) bytes of device scratch.
 *  opts->max_steps must be > 0: the call enqueues exactly that many step attempts per column and
 *  returns without synchronising; columns that reach t_bound earlier idle, the others come back with
 *  MARLPDE_STATUS_STEP_BUDGET and are resumed by calling again with the returned state.
 *  The host-pointer marlpde_rk45_integrate picks this path by itself when n_cells exceeds
 *  marlpde_rk45_max_cells() and repeats calls until every column has finished (or max_steps is used up).
 */
size_t marlpde_rk45_stream_workspace_bytes(int n_columns, int n_cells);
int marlpde_rk45_stream_integrate_dev(double* d_y, const marlpde_column_params* d_params,
                                      marlpde_column_state* d_state, int n_columns, int n_cells,
                                      const marlpde_rk45_options* opts, const double* d_t_eval,
                                      double* d_snapshots, void* d_workspace, size_t workspace_bytes,
                                      void* stream);
int marlpde_rk45_stream_integrate_events_dev(double* d_y, const marlpde_column_params* d_params,
                                             marlpde_column_state* d_state, int n_columns, int n_cells,
                                             const marlpde_rk45_options* opts, const double* d_t_eval,
                                             double* d_snapshots, int32_t* d_event_counts, double* d_event_times,
                                             void* d_workspace, size_t workspace_bytes, void* stream);

/* ---- batched implicit integrator: 3-stage Radau IIA with a block-tridiagonal simplified Newton solve
 * (replaces solve_ivp(method="Radau", jac_sparsity=...) per column; scipy/integrate/_ivp/radau.py) ------
 *  Arguments as for marlpde_rk45_integrate_dev (same options struct, same event outputs: with
 *  MARLPDE_FLAG_EVENTS the 7 monitors are evaluated after every accepted step and sign changes are
 *  located with Brent's method on the cubic Radau dense output), plus
 *  d_stats    [n_columns][4] int64, accumulated: Jacobian evaluations (njev), LU factorisations (nlu),
 *             Newton iterations, Newton failures
 *  d_workspace  marlpde_radau_workspace_bytes(n_columns, n_cells) bytes of device scratch (Jacobian
 *             blocks, factors and stage vectors of every column; need not be initialised)
 *  Any n_cells >= 3 is accepted (nothing has to fit on chip).  A column that stops on the step budget
 *  resumes "cold": (t, h_abs, y) are kept, the Jacobian and the Newton start guess are rebuilt.
 *  opts->quantum = K > 0 (TEAM columns): the first K columns of the batch — the longest ones of a cost-ordered sweep,
 *  whose sequential time bounds the whole sweep, or all columns of a small batch — are integrated by two warps each
 *  (a CTA per column: split RHS / element-wise passes / Jacobian, the two factorisation chains side by side), launched
 *  on an internal second stream next to the one-warp-per-column launch of the others and joined back into `stream`.
 *  d_queue must then hold TWO zeroed int32.  Same results up to the order of the norm reductions (1e-11).
 */
size_t marlpde_radau_workspace_bytes(int n_columns, int n_cells);
int marlpde_radau_integrate_dev(double* d_y, const marlpde_column_params* d_params,
                                marlpde_column_state* d_state, int n_columns, int n_cells,
                                const marlpde_rk45_options* opts, const double* d_t_eval,
                                double* d_snapshots, int32_t* d_event_counts, double* d_event_times,
                                int64_t* d_stats, void* d_workspace, size_t workspace_bytes,
                                int32_t* d_queue, void* stream);
int marlpde_radau_integrate(double* y, const marlpde_column_params* params,
                            marlpde_column_state* state, int n_columns, int n_cells,
                            const marlpde_rk45_options* opts, const double* t_eval,
                            double* snapshots, int32_t* event_counts, double* event_times,
                            int64_t* stats, int device);
/* stream-ordered variant, see marlpde_rk45_integrate_async */
int marlpde_radau_integrate_async(double* y, const marlpde_column_params* params,
                                  marlpde_column_state* state, int n_columns, int n_cells,
                                  const marlpde_rk45_options* opts, const double* t_eval,
                                  double* snapshots, int32_t* event_counts, double* event_times,
                                  int64_t* stats, int device, void* stream);

/* ---- batched implicit integrator: variable-order BDF (orders 1-5, NDF coefficients, quasi-constant step)
 * (replaces solve_ivp(method="BDF", jac_sparsity=...) per column — marlpde/parameters.py:213-216, :235-236;
 * scipy/integrate/_ivp/bdf.py — and is the device path for method="LSODA" batches, parameters.py:214-219: on this
 * stiff system LSODA runs in its BDF mode, see csrc/bdf_batch.cu) -----------------------------------------
 *  Arguments, outputs and statistics exactly as for marlpde_radau_integrate*; events are located with Brent's
 *  method on the BDF dense output (the step's differences array).  The workspace is
 *  marlpde_bdf_workspace_bytes(n_columns, n_cells).  A column that stops on the step budget resumes at
 *  order 1 from (t, h_abs, y): the differences array is not part of marlpde_column_state.
 */
size_t marlpde_bdf_workspace_bytes(int n_columns, int n_cells);
int marlpde_bdf_integrate_dev(double* d_y, const marlpde_column_params* d_params,
                              marlpde_column_state* d_state, int n_columns, int n_cells,
                              const marlpde_rk45_options* opts, const double* d_t_eval,
                              double* d_snapshots, int32_t* d_event_counts, double* d_event_times,
                              int64_t* d_stats, void* d_workspace, size_t workspace_bytes,
                              int32_t* d_queue, void* stream);
int marlpde_bdf_integrate(double* y, const marlpde_column_params* params,
                          marlpde_column_state* state, int n_columns, int n_cells,
                          const marlpde_rk45_options* opts, const double* t_eval,
                          double* snapshots, int32_t* event_counts, double* event_times,
                          int64_t* stats, int device);
int marlpde_bdf_integrate_async(double* y, const marlpde_column_params* params,
                                marlpde_column_state* state, int n_columns, int n_cells,
                                const marlpde_rk45_options* opts, const double* t_eval,
                                double* snapshots, int32_t* event_counts, double* event_times,
                                int64_t* stats, int device, void* stream);

/* ---- batched explicit Runge-Kutta integrators: Bogacki-Shampine RK23 and Dormand-Prince DOP853
 * (replace solve_ivp(method="RK23" | "DOP853") per column — marlpde/parameters.py:213; scipy/integrate/_ivp/rk.py —
 * step for step: same tableaux, step-size control, error norms and dense output, see csrc/erk_batch.cu) ------------
 *  Arguments and outputs as for marlpde_bdf_integrate* without the statistics: same options struct (opts->quantum
 *  must be 0), same column state and status codes; t_eval samples and events use each method's dense output (DOP853:
 *  the three extra stages are evaluated, and counted in nfev, only in steps that sample t_eval or locate an event).
 *  The workspace is marlpde_{rk23,dop853}_workspace_bytes(n_columns, n_cells); d_queue is one zeroed int32.  Any
 *  n_cells >= 3.  A column that stops on the step budget stops after an accepted step and resumes from (t, h_abs, y)
 *  bit-identically (nfev counts one extra evaluation of f(y) per resume).
 */
size_t marlpde_rk23_workspace_bytes(int n_columns, int n_cells);
int marlpde_rk23_integrate_dev(double* d_y, const marlpde_column_params* d_params,
                               marlpde_column_state* d_state, int n_columns, int n_cells,
                               const marlpde_rk45_options* opts, const double* d_t_eval,
                               double* d_snapshots, int32_t* d_event_counts, double* d_event_times,
                               void* d_workspace, size_t workspace_bytes, int32_t* d_queue, void* stream);
int marlpde_rk23_integrate(double* y, const marlpde_column_params* params,
                           marlpde_column_state* state, int n_columns, int n_cells,
                           const marlpde_rk45_options* opts, const double* t_eval,
                           double* snapshots, int32_t* event_counts, double* event_times, int device);
int marlpde_rk23_integrate_async(double* y, const marlpde_column_params* params,
                                 marlpde_column_state* state, int n_columns, int n_cells,
                                 const marlpde_rk45_options* opts, const double* t_eval,
                                 double* snapshots, int32_t* event_counts, double* event_times,
                                 int device, void* stream);
size_t marlpde_dop853_workspace_bytes(int n_columns, int n_cells);
int marlpde_dop853_integrate_dev(double* d_y, const marlpde_column_params* d_params,
                                 marlpde_column_state* d_state, int n_columns, int n_cells,
                                 const marlpde_rk45_options* opts, const double* d_t_eval,
                                 double* d_snapshots, int32_t* d_event_counts, double* d_event_times,
                                 void* d_workspace, size_t workspace_bytes, int32_t* d_queue, void* stream);
int marlpde_dop853_integrate(double* y, const marlpde_column_params* params,
                             marlpde_column_state* state, int n_columns, int n_cells,
                             const marlpde_rk45_options* opts, const double* t_eval,
                             double* snapshots, int32_t* event_counts, double* event_times, int device);
int marlpde_dop853_integrate_async(double* y, const marlpde_column_params* params,
                                   marlpde_column_state* state, int n_columns, int n_cells,
                                   const marlpde_rk45_options* opts, const double* t_eval,
                                   double* snapshots, int32_t* event_counts, double* event_times,
                                   int device, void* stream);

/* ---- measurement helper: fp64 FMA peak (TFLOP/s, best of `repeats`) of `device`, the roofline
 * denominator of the fp64-pipe-bound RK45 kernel (no reference counterpart). */
int marlpde_probe_fp64_peak(int device, int iters, int repeats, double* tflops);
/* test helper: element-wise evaluation of the kernels' own fp64 maths (csrc/fp64_math.cuh) on HOST
 * arrays: op 0 log, 1 exp, 2 expm1, 3 reciprocal, 4 (1+x)/x, 5 Fiadeiro-Veronis coth(x)-1/x. */
int marlpde_probe_math(int op, const double* x, int n, double* out, int device);
/* test helper: the block-tridiagonal Jacobian the implicit kernels use (analytic 5x5 blocks), for ONE column
 * on HOST arrays: y [5][n_cells] field-major, J_out [n_cells][3][5][5] = blocks L, D, U of every cell, each
 * stored [column][row]. */
int marlpde_probe_jacobian(const double* y, const marlpde_column_params* params, int n_cells, double* J_out,
                           int device);

#ifdef __cplusplus
}
#endif
#endif /* MARLPDE_B200_H */
