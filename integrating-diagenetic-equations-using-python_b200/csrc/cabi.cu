// cabi.cu — the extern "C" boundary declared in include/marlpde_b200.h.
// Host-pointer entry points stage through device memory and synchronise; *_dev entry points
// only enqueue work on the caller's stream.  There is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>

#include <chrono>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/marlpde_b200.h"
#include "bdf_batch.cuh"
#include "erk_batch.cuh"
#include "radau_batch.cuh"
#include "rk45_persistent.cuh"
#include "rk45_streaming.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int cuda_fail(cudaError_t e, const char* what) {
  return fail(MARLPDE_ECUDA, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
}

#define CU(call)                                         \
  do {                                                   \
    cudaError_t e_ = (call);                             \
    if (e_ != cudaSuccess) return cuda_fail(e_, #call);  \
  } while (0)

struct DevProps {
  int sm_count = 0;
  int smem_optin = 0;
  bool ok = false;
};

int current_props(DevProps& p) {
  int dev = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&p.sm_count, cudaDevAttrMultiProcessorCount, dev));
  CU(cudaDeviceGetAttribute(&p.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  p.ok = true;
  return MARLPDE_OK;
}

// MARLPDE_TRACE=1: wall-clock phases of the host-pointer entry points on stderr (the reference prints
// the wall time around solve_ivp, Evolve_scenario.py:90, :110, :148-149)
struct PhaseTrace {
  bool on;
  const char* what;
  std::chrono::steady_clock::time_point t0;
  explicit PhaseTrace(const char* w) : on(std::getenv("MARLPDE_TRACE") != nullptr), what(w), t0(std::chrono::steady_clock::now()) {}
  void mark(const char* phase) {
    if (!on) return;
    const auto t1 = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[marlpde trace] %s: %-10s %8.2f ms\n", what, phase,
                 std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};

// Device scratch of the host-pointer entry points comes from one stream-ordered memory pool per device
// (cudaMallocFromPoolAsync / cudaFreeAsync): allocation and release are enqueued on the call's stream like the copies and
// the kernel, so the *_async entry points return without synchronising, and blocks are reused from call to call
// (cudaMalloc / cudaFree cost 3-130 ms per call on the bench box, r01c).  The pool keeps at most kPoolKeepBytes
// cached between calls (release threshold; anything above goes back to the driver at the next synchronisation), so a
// sweep with a large snapshot buffer does not park gigabytes next to the caller's own allocator;
// marlpde_release_cached_memory() trims it to zero.
constexpr unsigned long long kPoolKeepBytes = 256ull << 20;
std::mutex g_pool_mutex;
cudaMemPool_t g_pools[64] = {};

cudaError_t pool_for(int device, cudaMemPool_t* out) {
  if (device < 0 || device >= 64) return cudaErrorInvalidDevice;
  std::lock_guard<std::mutex> lock(g_pool_mutex);
  if (!g_pools[device]) {
    cudaMemPoolProps props;
    std::memset(&props, 0, sizeof props);
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device;
    cudaError_t e = cudaMemPoolCreate(&g_pools[device], &props);
    if (e != cudaSuccess) return e;
    unsigned long long keep = kPoolKeepBytes;
    e = cudaMemPoolSetAttribute(g_pools[device], cudaMemPoolAttrReleaseThreshold, &keep);
    if (e != cudaSuccess) return e;
  }
  *out = g_pools[device];
  return cudaSuccess;
}

struct DevBuf {            // freed in stream order when it goes out of scope (after everything enqueued before)
  void* p = nullptr;
  cudaStream_t stream = nullptr;
  ~DevBuf() {
    if (p) cudaFreeAsync(p, stream);
  }
  cudaError_t alloc(size_t n, cudaStream_t s) {
    if (n == 0) n = 1;
    int device = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e != cudaSuccess) return e;
    cudaMemPool_t pool;
    e = pool_for(device, &pool);
    if (e != cudaSuccess) return e;
    stream = s;
    e = cudaMallocFromPoolAsync(&p, n, pool, s);
    if (e != cudaSuccess) p = nullptr;
    return e;
  }
  template <typename T> T* as() { return static_cast<T*>(p); }
};

// The host-pointer entry points run on `device` and leave the calling thread's current device as they found it
// (a multi-GPU caller's torch.cuda.current_device() must not change behind its back).
struct DeviceScope {
  int prev = -1;
  bool changed = false;
  ~DeviceScope() {
    if (changed) cudaSetDevice(prev);
  }
  int enter(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
      return fail(MARLPDE_ENODEVICE, "no CUDA device available (%s); this library has no CPU path",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(MARLPDE_EINVAL, "device %d out of range [0,%d)", device, n);
    CU(cudaGetDevice(&prev));
    if (prev != device) {
      CU(cudaSetDevice(device));
      changed = true;
    }
    return MARLPDE_OK;
  }
};

// MARLPDE_FLAG_* bits implied by the model variants present in a HOST params array
int model_flags_of(const marlpde_column_params* params, int n_columns) {
  for (int c = 0; c < n_columns; ++c)
    if (params[c].model_flags & MARLPDE_MODEL_VAR_DPHI) return (int)MARLPDE_FLAG_VAR_DPHI;
  return 0;
}

}  // namespace

extern "C" {

int marlpde_abi_version(void) { return MARLPDE_ABI_VERSION; }

int marlpde_struct_size(int which) {
  switch (which) {
    case 0: return (int)sizeof(marlpde_column_params);
    case 1: return (int)sizeof(marlpde_rk45_options);
    case 2: return (int)sizeof(marlpde_column_state);
    case 3: return (int)sizeof(marlpde_device_info);
    default: return -1;
  }
}

const char* marlpde_last_error(void) { return g_err; }

int marlpde_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int marlpde_get_device_info(int device, marlpde_device_info* info) {
  if (!info) return fail(MARLPDE_EINVAL, "info is NULL");
  int n = marlpde_device_count();
  if (n == 0) return fail(MARLPDE_ENODEVICE, "no CUDA device available");
  if (device < 0 || device >= n) return fail(MARLPDE_EINVAL, "device %d out of range [0,%d)", device, n);
  cudaDeviceProp p;
  CU(cudaGetDeviceProperties(&p, device));
  std::memset(info, 0, sizeof(*info));
  std::strncpy(info->name, p.name, sizeof(info->name) - 1);
  info->sm_count = p.multiProcessorCount;
  info->cc_major = p.major;
  info->cc_minor = p.minor;
  info->max_smem_per_block = (int32_t)p.sharedMemPerBlockOptin;
  info->total_mem = (int64_t)p.totalGlobalMem;
  return MARLPDE_OK;
}

int marlpde_release_cached_memory(void) {
  std::lock_guard<std::mutex> lock(g_pool_mutex);
  int n = 0;
  for (int d = 0; d < 64; ++d)
    if (g_pools[d]) {
      cudaMemPoolTrimTo(g_pools[d], 0);
      ++n;
    }
  return n;
}

int marlpde_rk45_max_cells(void) { return marlpde::rk45_max_cells(); }

int marlpde_rk45_columns_per_cta(int n_cells) {
  // 227 KB is the sm_100 opt-in limit per CTA; the launcher re-checks against the real device.
  return marlpde::rk45_columns_per_cta(n_cells, 227 * 1024);
}

int marlpde_rhs_batch_dev(const double* d_y, const marlpde_column_params* d_params, int n_columns,
                          int n_cells, double* d_out, void* stream) {
  if (n_columns < 0 || n_cells < 2) return fail(MARLPDE_EINVAL, "need n_columns >= 0 and n_cells >= 2");
  if (n_columns == 0) return MARLPDE_OK;
  if (!d_y || !d_params || !d_out) return fail(MARLPDE_EINVAL, "NULL device pointer");
  cudaError_t e = marlpde::launch_rhs_batch(d_y, d_params, n_columns, n_cells, d_out, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "rhs_batch launch");
  return MARLPDE_OK;
}

int marlpde_rhs_batch(const double* y, const marlpde_column_params* params, int n_columns, int n_cells,
                      double* out, int device) {
  if (n_columns < 0 || n_cells < 2) return fail(MARLPDE_EINVAL, "need n_columns >= 0 and n_cells >= 2");
  if (n_columns == 0) return MARLPDE_OK;
  if (!y || !params || !out) return fail(MARLPDE_EINVAL, "NULL pointer");
  DeviceScope scope;
  int rc = scope.enter(device);
  if (rc) return rc;
  cudaStream_t s = cudaStreamPerThread;
  const size_t nb = sizeof(double) * 5 * (size_t)n_cells * n_columns;
  const size_t nb_p = sizeof(marlpde_column_params) * (size_t)n_columns;
  DevBuf dy, dp, dout;
  CU(dy.alloc(nb, s));
  CU(dout.alloc(nb, s));
  CU(dp.alloc(nb_p, s));
  CU(cudaMemcpyAsync(dy.p, y, nb, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dp.p, params, nb_p, cudaMemcpyHostToDevice, s));
  rc = marlpde_rhs_batch_dev(dy.as<double>(), dp.as<marlpde_column_params>(), n_columns, n_cells, dout.as<double>(), s);
  if (rc) return rc;
  CU(cudaMemcpyAsync(out, dout.p, nb, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return MARLPDE_OK;
}

static int check_rk45_args(int n_columns, int n_cells, const marlpde_rk45_options* opts) {
  if (!opts) return fail(MARLPDE_EINVAL, "opts is NULL");
  if (n_columns < 0) return fail(MARLPDE_EINVAL, "n_columns < 0");
  if (n_cells < 32 || n_cells > marlpde::rk45_max_cells())
    return fail(MARLPDE_EUNSUPPORTED, "on-chip RK45 kernel supports 32 <= n_cells <= %d (got %d)",
                marlpde::rk45_max_cells(), n_cells);
  if (!(opts->rtol > 0.0) || !(opts->atol >= 0.0)) return fail(MARLPDE_EINVAL, "need rtol > 0, atol >= 0");
  if (!(opts->max_step > 0.0)) return fail(MARLPDE_EINVAL, "max_step must be positive (use +inf for none)");
  if (opts->n_eval < 0 || opts->event_capacity < 0) return fail(MARLPDE_EINVAL, "negative n_eval/event_capacity");
  return MARLPDE_OK;
}

int marlpde_rk45_integrate_dev(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                               int n_columns, int n_cells, const marlpde_rk45_options* opts,
                               const double* d_t_eval, double* d_snapshots, int32_t* d_event_counts,
                               double* d_event_times, int32_t* d_queue, void* stream) {
  int rc = check_rk45_args(n_columns, n_cells, opts);
  if (rc) return rc;
  if (n_columns == 0) return MARLPDE_OK;
  if (!d_y || !d_params || !d_state || !d_queue) return fail(MARLPDE_EINVAL, "NULL device pointer");
  if (opts->n_eval > 0 && (!d_t_eval || !d_snapshots)) return fail(MARLPDE_EINVAL, "n_eval > 0 needs t_eval and snapshots");
  marlpde_rk45_options o = *opts;
  if (o.flags & MARLPDE_FLAG_EVENTS) {
    if (!d_event_counts) return fail(MARLPDE_EINVAL, "MARLPDE_FLAG_EVENTS needs event_counts");
    if (o.event_capacity > 0 && !d_event_times) return fail(MARLPDE_EINVAL, "event_capacity > 0 needs event_times");
  }
  DevProps props;
  rc = current_props(props);
  if (rc) return rc;
  if (marlpde::rk45_columns_per_cta(n_cells, props.smem_optin) <= 0)
    return fail(MARLPDE_EUNSUPPORTED, "n_cells=%d does not fit %d bytes of shared memory", n_cells, props.smem_optin);
  cudaError_t e = marlpde::launch_rk45(d_y, d_params, d_state, n_columns, n_cells, o, d_t_eval, d_snapshots,
                                       d_event_counts, d_event_times, d_queue, props.sm_count, props.smem_optin, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "rk45 launch");
  return MARLPDE_OK;
}

static int check_stream_args(int n_columns, int n_cells, const marlpde_rk45_options* opts);
extern "C" int marlpde_rk45_stream_integrate_events_dev(double*, const marlpde_column_params*, marlpde_column_state*, int, int,
                                                        const marlpde_rk45_options*, const double*, double*, int32_t*,
                                                        double*, void*, size_t, void*);

// Host-pointer driver of the streaming path: repeats fixed-size batches of step attempts until every
// column has left the STEP_BUDGET state (or the caller's max_steps budget is used up).  The per-batch status
// read-back makes it synchronous by nature.
static int rk45_integrate_streaming(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                                    int n_columns, int n_cells, const marlpde_rk45_options* opts,
                                    const double* t_eval, double* snapshots, int32_t* event_counts, double* event_times,
                                    int device, cudaStream_t s) {
  int rc = check_stream_args(n_columns, n_cells, opts);
  if (rc) return rc;
  if (n_columns == 0) return MARLPDE_OK;
  if (!y || !params || !state) return fail(MARLPDE_EINVAL, "NULL pointer");
  if (opts->n_eval > 0 && (!t_eval || !snapshots)) return fail(MARLPDE_EINVAL, "n_eval > 0 needs t_eval and snapshots");
  DeviceScope scope;
  rc = scope.enter(device);
  if (rc) return rc;
  const size_t nb_y = sizeof(double) * 5 * (size_t)n_cells * n_columns;
  const size_t nb_snap = nb_y * (size_t)opts->n_eval;
  const size_t nb_state = sizeof(marlpde_column_state) * (size_t)n_columns;
  const size_t nb_p = sizeof(marlpde_column_params) * (size_t)n_columns;
  const size_t nb_work = marlpde::rk45_stream_workspace_bytes(n_columns, n_cells);
  const bool ev = (opts->flags & MARLPDE_FLAG_EVENTS) != 0;
  const size_t nb_ec = sizeof(int32_t) * MARLPDE_NEVENTS * (size_t)n_columns;
  const size_t nb_et = sizeof(double) * MARLPDE_NEVENTS * (size_t)(opts->event_capacity > 0 ? opts->event_capacity : 0) * n_columns;
  DevBuf dy, dp, ds, dte, dsnap, dw, dec, det;
  CU(dy.alloc(nb_y, s));
  CU(dp.alloc(nb_p, s));
  CU(ds.alloc(nb_state, s));
  CU(dte.alloc(sizeof(double) * (size_t)opts->n_eval, s));
  CU(dsnap.alloc(nb_snap, s));
  CU(dw.alloc(nb_work, s));
  CU(dec.alloc(nb_ec, s));
  CU(det.alloc(nb_et, s));
  CU(cudaMemcpyAsync(dy.p, y, nb_y, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dp.p, params, nb_p, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(ds.p, state, nb_state, cudaMemcpyHostToDevice, s));
  if (opts->n_eval) CU(cudaMemcpyAsync(dte.p, t_eval, sizeof(double) * (size_t)opts->n_eval, cudaMemcpyHostToDevice, s));
  if (snapshots && nb_snap) CU(cudaMemcpyAsync(dsnap.p, snapshots, nb_snap, cudaMemcpyHostToDevice, s));
  if (ev) {
    if (event_counts) CU(cudaMemcpyAsync(dec.p, event_counts, nb_ec, cudaMemcpyHostToDevice, s));
    else CU(cudaMemsetAsync(dec.p, 0, nb_ec, s));
    if (event_times && nb_et) CU(cudaMemcpyAsync(det.p, event_times, nb_et, cudaMemcpyHostToDevice, s));
  }
  const long long budget = opts->max_steps > 0 ? opts->max_steps : -1;   // -1: until done
  long long used = 0;
  std::vector<marlpde_column_state> hs((size_t)n_columns);
  for (;;) {
    marlpde_rk45_options o = *opts;
    o.flags |= model_flags_of(params, n_columns);
    long long batch = 512;
    if (budget > 0 && budget - used < batch) batch = budget - used;
    o.max_steps = batch;
    rc = marlpde_rk45_stream_integrate_events_dev(dy.as<double>(), dp.as<marlpde_column_params>(),
                                                  ds.as<marlpde_column_state>(), n_columns, n_cells, &o, dte.as<double>(),
                                                  dsnap.as<double>(), ev ? dec.as<int32_t>() : nullptr,
                                                  ev ? det.as<double>() : nullptr, dw.p, nb_work, s);
    if (rc) return rc;
    CU(cudaMemcpyAsync(hs.data(), ds.p, nb_state, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    used += batch;
    bool pending = false;
    for (int c = 0; c < n_columns; ++c)
      pending = pending || hs[(size_t)c].status == MARLPDE_STATUS_STEP_BUDGET ||
                hs[(size_t)c].status == MARLPDE_STATUS_STEP_BUDGET_MIDSTEP;
    if (!pending || (budget > 0 && used >= budget)) break;
  }
  CU(cudaMemcpyAsync(y, dy.p, nb_y, cudaMemcpyDeviceToHost, s));
  std::memcpy(state, hs.data(), nb_state);
  if (snapshots && nb_snap) CU(cudaMemcpyAsync(snapshots, dsnap.p, nb_snap, cudaMemcpyDeviceToHost, s));
  if (ev && event_counts) CU(cudaMemcpyAsync(event_counts, dec.p, nb_ec, cudaMemcpyDeviceToHost, s));
  if (ev && event_times && nb_et) CU(cudaMemcpyAsync(event_times, det.p, nb_et, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return MARLPDE_OK;
}

// H2D of the inputs, one launch, D2H of the results, all enqueued on `s`; synchronises only if `sync`.
static int rk45_integrate_host(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                               int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* t_eval,
                               double* snapshots, int32_t* event_counts, double* event_times, int device,
                               cudaStream_t s, bool sync) {
  if (opts && (n_cells > marlpde::rk45_max_cells() || (n_cells >= 2 && n_cells < 32)))
    return rk45_integrate_streaming(y, params, state, n_columns, n_cells, opts, t_eval, snapshots, event_counts,
                                    event_times, device, s);
  int rc = check_rk45_args(n_columns, n_cells, opts);
  if (rc) return rc;
  if (n_columns == 0) return MARLPDE_OK;
  if (!y || !params || !state) return fail(MARLPDE_EINVAL, "NULL pointer");
  if (opts->n_eval > 0 && (!t_eval || !snapshots)) return fail(MARLPDE_EINVAL, "n_eval > 0 needs t_eval and snapshots");
  DeviceScope scope;
  rc = scope.enter(device);
  if (rc) return rc;
  const size_t nb_y = sizeof(double) * 5 * (size_t)n_cells * n_columns;
  const size_t nb_snap = nb_y * (size_t)opts->n_eval;
  const size_t nb_p = sizeof(marlpde_column_params) * (size_t)n_columns;
  const size_t nb_s = sizeof(marlpde_column_state) * (size_t)n_columns;
  const size_t nb_ec = sizeof(int32_t) * MARLPDE_NEVENTS * (size_t)n_columns;
  const size_t nb_et = sizeof(double) * MARLPDE_NEVENTS * (size_t)opts->event_capacity * n_columns;
  PhaseTrace trace("rk45_integrate");
  DevBuf dy, dp, ds, dte, dsnap, dq, dec, det;
  CU(dy.alloc(nb_y, s));
  CU(dp.alloc(nb_p, s));
  CU(ds.alloc(nb_s, s));
  CU(dte.alloc(sizeof(double) * (size_t)opts->n_eval, s));
  CU(dsnap.alloc(nb_snap, s));
  const size_t nb_q = sizeof(int32_t) * (1 + 2 * (size_t)n_columns);   // work counter + lock word and attempt counter per column
  CU(dq.alloc(nb_q, s));
  CU(dec.alloc(nb_ec, s));
  CU(det.alloc(nb_et, s));
  trace.mark("alloc");
  CU(cudaMemcpyAsync(dy.p, y, nb_y, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dp.p, params, nb_p, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(ds.p, state, nb_s, cudaMemcpyHostToDevice, s));
  if (opts->n_eval) CU(cudaMemcpyAsync(dte.p, t_eval, sizeof(double) * (size_t)opts->n_eval, cudaMemcpyHostToDevice, s));
  if (snapshots && nb_snap) CU(cudaMemcpyAsync(dsnap.p, snapshots, nb_snap, cudaMemcpyHostToDevice, s));
  CU(cudaMemsetAsync(dq.p, 0, nb_q, s));
  if (event_counts) CU(cudaMemcpyAsync(dec.p, event_counts, nb_ec, cudaMemcpyHostToDevice, s));
  else CU(cudaMemsetAsync(dec.p, 0, nb_ec, s));
  if (event_times && nb_et) CU(cudaMemcpyAsync(det.p, event_times, nb_et, cudaMemcpyHostToDevice, s));
  marlpde_rk45_options o = *opts;
  o.flags |= MARLPDE_FLAG_QUEUE_LOCKS | model_flags_of(params, n_columns);
  rc = marlpde_rk45_integrate_dev(dy.as<double>(), dp.as<marlpde_column_params>(), ds.as<marlpde_column_state>(),
                                  n_columns, n_cells, &o, dte.as<double>(), dsnap.as<double>(),
                                  dec.as<int32_t>(), det.as<double>(), dq.as<int32_t>(), s);
  if (rc) return rc;
  trace.mark("h2d+launch");
  if (trace.on) {
    CU(cudaStreamSynchronize(s));
    trace.mark("kernel");
  }
  CU(cudaMemcpyAsync(y, dy.p, nb_y, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(state, ds.p, nb_s, cudaMemcpyDeviceToHost, s));
  if (snapshots && nb_snap) CU(cudaMemcpyAsync(snapshots, dsnap.p, nb_snap, cudaMemcpyDeviceToHost, s));
  if (event_counts) CU(cudaMemcpyAsync(event_counts, dec.p, nb_ec, cudaMemcpyDeviceToHost, s));
  if (event_times && nb_et) CU(cudaMemcpyAsync(event_times, det.p, nb_et, cudaMemcpyDeviceToHost, s));
  if (sync) CU(cudaStreamSynchronize(s));
  trace.mark("d2h");
  return MARLPDE_OK;
}

int marlpde_rk45_integrate(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                           int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* t_eval,
                           double* snapshots, int32_t* event_counts, double* event_times, int device) {
  return rk45_integrate_host(y, params, state, n_columns, n_cells, opts, t_eval, snapshots, event_counts, event_times,
                             device, cudaStreamPerThread, true);
}

int marlpde_rk45_integrate_async(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                                 int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* t_eval,
                                 double* snapshots, int32_t* event_counts, double* event_times, int device,
                                 void* stream) {
  return rk45_integrate_host(y, params, state, n_columns, n_cells, opts, t_eval, snapshots, event_counts, event_times,
                             device, (cudaStream_t)stream, false);
}

size_t marlpde_rk45_stream_workspace_bytes(int n_columns, int n_cells) {
  if (n_columns <= 0 || n_cells <= 0) return 0;
  return marlpde::rk45_stream_workspace_bytes(n_columns, n_cells);
}

static int check_stream_args(int n_columns, int n_cells, const marlpde_rk45_options* opts) {
  if (!opts) return fail(MARLPDE_EINVAL, "opts is NULL");
  if (n_columns < 0) return fail(MARLPDE_EINVAL, "n_columns < 0");
  if (n_cells < 2) return fail(MARLPDE_EINVAL, "need n_cells >= 2");
  if (!(opts->rtol > 0.0) || !(opts->atol >= 0.0)) return fail(MARLPDE_EINVAL, "need rtol > 0, atol >= 0");
  if (!(opts->max_step > 0.0)) return fail(MARLPDE_EINVAL, "max_step must be positive (use +inf for none)");
  if (opts->n_eval < 0) return fail(MARLPDE_EINVAL, "negative n_eval");
  if (opts->n_eval < 0 || opts->event_capacity < 0) return fail(MARLPDE_EINVAL, "negative n_eval/event_capacity");
  return MARLPDE_OK;
}

int marlpde_rk45_stream_integrate_events_dev(double* d_y, const marlpde_column_params* d_params,
                                             marlpde_column_state* d_state, int n_columns, int n_cells,
                                             const marlpde_rk45_options* opts, const double* d_t_eval,
                                             double* d_snapshots, int32_t* d_event_counts, double* d_event_times,
                                             void* d_workspace, size_t workspace_bytes, void* stream) {
  int rc = check_stream_args(n_columns, n_cells, opts);
  if (rc) return rc;
  if (n_columns == 0) return MARLPDE_OK;
  if (opts->max_steps <= 0) return fail(MARLPDE_EINVAL, "the streaming path needs max_steps > 0 per call");
  if (opts->max_steps > 1000000) return fail(MARLPDE_EINVAL, "max_steps per call is limited to 1e6 on the streaming path");
  if (!d_y || !d_params || !d_state || !d_workspace) return fail(MARLPDE_EINVAL, "NULL device pointer");
  if (opts->n_eval > 0 && (!d_t_eval || !d_snapshots)) return fail(MARLPDE_EINVAL, "n_eval > 0 needs t_eval and snapshots");
  if (opts->flags & MARLPDE_FLAG_EVENTS) {
    if (!d_event_counts) return fail(MARLPDE_EINVAL, "MARLPDE_FLAG_EVENTS needs event_counts");
    if (opts->event_capacity > 0 && !d_event_times) return fail(MARLPDE_EINVAL, "event_capacity > 0 needs event_times");
  }
  if (workspace_bytes < marlpde::rk45_stream_workspace_bytes(n_columns, n_cells))
    return fail(MARLPDE_EINVAL, "workspace too small: %zu < %zu bytes", workspace_bytes,
                marlpde::rk45_stream_workspace_bytes(n_columns, n_cells));
  cudaError_t e = marlpde::launch_rk45_stream(d_y, d_params, d_state, n_columns, n_cells, *opts, d_t_eval,
                                              d_snapshots, d_event_counts, d_event_times, d_workspace, opts->max_steps,
                                              (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "rk45 stream launch");
  return MARLPDE_OK;
}

int marlpde_rk45_stream_integrate_dev(double* d_y, const marlpde_column_params* d_params,
                                      marlpde_column_state* d_state, int n_columns, int n_cells,
                                      const marlpde_rk45_options* opts, const double* d_t_eval, double* d_snapshots,
                                      void* d_workspace, size_t workspace_bytes, void* stream) {
  if (opts && (opts->flags & MARLPDE_FLAG_EVENTS))
    return fail(MARLPDE_EINVAL, "MARLPDE_FLAG_EVENTS: call marlpde_rk45_stream_integrate_events_dev (it takes the event outputs)");
  return marlpde_rk45_stream_integrate_events_dev(d_y, d_params, d_state, n_columns, n_cells, opts, d_t_eval, d_snapshots,
                                                  nullptr, nullptr, d_workspace, workspace_bytes, stream);
}

// ---- implicit integrators: the Radau IIA and the BDF kernel share arguments, buffers and checks ----------------------
enum ImplicitKind { kRadau = 0, kBdf = 1 };

static size_t implicit_workspace_bytes(ImplicitKind kind, int n_columns, int n_cells) {
  return kind == kRadau ? marlpde::radau_workspace_bytes(n_columns, n_cells)
                        : marlpde::bdf_workspace_bytes(n_columns, n_cells);
}

size_t marlpde_radau_workspace_bytes(int n_columns, int n_cells) {
  if (n_columns <= 0 || n_cells <= 0) return 0;
  return implicit_workspace_bytes(kRadau, n_columns, n_cells);
}

size_t marlpde_bdf_workspace_bytes(int n_columns, int n_cells) {
  if (n_columns <= 0 || n_cells <= 0) return 0;
  return implicit_workspace_bytes(kBdf, n_columns, n_cells);
}

static int check_implicit_args(int n_columns, int n_cells, const marlpde_rk45_options* opts) {
  if (!opts) return fail(MARLPDE_EINVAL, "opts is NULL");
  if (n_columns < 0) return fail(MARLPDE_EINVAL, "n_columns < 0");
  if (n_cells < 3) return fail(MARLPDE_EINVAL, "the implicit integrators need n_cells >= 3 (got %d)", n_cells);
  if (!(opts->rtol > 0.0) || !(opts->atol >= 0.0)) return fail(MARLPDE_EINVAL, "need rtol > 0, atol >= 0");
  if (!(opts->max_step > 0.0)) return fail(MARLPDE_EINVAL, "max_step must be positive (use +inf for none)");
  if (opts->n_eval < 0) return fail(MARLPDE_EINVAL, "negative n_eval");
  return MARLPDE_OK;
}

static int implicit_integrate_dev(ImplicitKind kind, double* d_y, const marlpde_column_params* d_params,
                                  marlpde_column_state* d_state, int n_columns, int n_cells,
                                  const marlpde_rk45_options* opts, const double* d_t_eval, double* d_snapshots,
                                  int32_t* d_event_counts, double* d_event_times, int64_t* d_stats, void* d_workspace,
                                  size_t workspace_bytes, int32_t* d_queue, void* stream) {
  int rc = check_implicit_args(n_columns, n_cells, opts);
  if (rc) return rc;
  if (n_columns == 0) return MARLPDE_OK;
  if (!d_y || !d_params || !d_state || !d_queue || !d_stats || !d_workspace)
    return fail(MARLPDE_EINVAL, "NULL device pointer");
  if (opts->n_eval > 0 && (!d_t_eval || !d_snapshots)) return fail(MARLPDE_EINVAL, "n_eval > 0 needs t_eval and snapshots");
  if (opts->flags & MARLPDE_FLAG_EVENTS) {
    if (!d_event_counts) return fail(MARLPDE_EINVAL, "MARLPDE_FLAG_EVENTS needs event_counts");
    if (opts->event_capacity > 0 && !d_event_times) return fail(MARLPDE_EINVAL, "event_capacity > 0 needs event_times");
  }
  if (opts->quantum < 0) return fail(MARLPDE_EINVAL, "negative quantum (team columns)");
  if (kind == kBdf && opts->quantum != 0) return fail(MARLPDE_EUNSUPPORTED, "team columns (opts->quantum) are a Radau feature");
  const size_t need = implicit_workspace_bytes(kind, n_columns, n_cells);
  if (workspace_bytes < need) return fail(MARLPDE_EINVAL, "workspace too small: %zu < %zu bytes", workspace_bytes, need);
  DevProps props;
  rc = current_props(props);
  if (rc) return rc;
  auto launch = kind == kRadau ? marlpde::launch_radau : marlpde::launch_bdf;
  cudaError_t e = launch(d_y, d_params, d_state, n_columns, n_cells, *opts, d_t_eval, d_snapshots, d_stats,
                         d_event_counts, d_event_times, static_cast<double*>(d_workspace), d_queue, props.sm_count,
                         (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, kind == kRadau ? "radau launch" : "bdf launch");
  return MARLPDE_OK;
}

int marlpde_radau_integrate_dev(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                                int n_columns, int n_cells, const marlpde_rk45_options* opts,
                                const double* d_t_eval, double* d_snapshots, int32_t* d_event_counts,
                                double* d_event_times, int64_t* d_stats, void* d_workspace, size_t workspace_bytes,
                                int32_t* d_queue, void* stream) {
  return implicit_integrate_dev(kRadau, d_y, d_params, d_state, n_columns, n_cells, opts, d_t_eval, d_snapshots,
                                d_event_counts, d_event_times, d_stats, d_workspace, workspace_bytes, d_queue, stream);
}

int marlpde_bdf_integrate_dev(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                              int n_columns, int n_cells, const marlpde_rk45_options* opts,
                              const double* d_t_eval, double* d_snapshots, int32_t* d_event_counts,
                              double* d_event_times, int64_t* d_stats, void* d_workspace, size_t workspace_bytes,
                              int32_t* d_queue, void* stream) {
  return implicit_integrate_dev(kBdf, d_y, d_params, d_state, n_columns, n_cells, opts, d_t_eval, d_snapshots,
                                d_event_counts, d_event_times, d_stats, d_workspace, workspace_bytes, d_queue, stream);
}

static int implicit_integrate_host(ImplicitKind kind, double* y, const marlpde_column_params* params,
                                   marlpde_column_state* state, int n_columns, int n_cells,
                                   const marlpde_rk45_options* opts, const double* t_eval, double* snapshots,
                                   int32_t* event_counts, double* event_times, int64_t* stats, int device,
                                   cudaStream_t s, bool sync) {
  int rc = check_implicit_args(n_columns, n_cells, opts);
  if (rc) return rc;
  if (n_columns == 0) return MARLPDE_OK;
  if (!y || !params || !state || !stats) return fail(MARLPDE_EINVAL, "NULL pointer");
  if (opts->n_eval > 0 && (!t_eval || !snapshots)) return fail(MARLPDE_EINVAL, "n_eval > 0 needs t_eval and snapshots");
  DeviceScope scope;
  rc = scope.enter(device);
  if (rc) return rc;
  const size_t nb_y = sizeof(double) * 5 * (size_t)n_cells * n_columns;
  const size_t nb_snap = nb_y * (size_t)opts->n_eval;
  const size_t nb_p = sizeof(marlpde_column_params) * (size_t)n_columns;
  const size_t nb_s = sizeof(marlpde_column_state) * (size_t)n_columns;
  const size_t nb_stats = sizeof(int64_t) * 4 * (size_t)n_columns;
  const size_t nb_work = implicit_workspace_bytes(kind, n_columns, n_cells);
  const size_t nb_ec = sizeof(int32_t) * MARLPDE_NEVENTS * (size_t)n_columns;
  const size_t nb_et = sizeof(double) * MARLPDE_NEVENTS * (size_t)(opts->event_capacity > 0 ? opts->event_capacity : 0) * n_columns;
  DevBuf dy, dp, ds, dte, dsnap, dq, dst, dw, dec, det;
  CU(dec.alloc(nb_ec, s));
  CU(det.alloc(nb_et, s));
  if (event_counts) CU(cudaMemcpyAsync(dec.p, event_counts, nb_ec, cudaMemcpyHostToDevice, s));
  else CU(cudaMemsetAsync(dec.p, 0, nb_ec, s));
  if (event_times && nb_et) CU(cudaMemcpyAsync(det.p, event_times, nb_et, cudaMemcpyHostToDevice, s));
  CU(dy.alloc(nb_y, s));
  CU(dp.alloc(nb_p, s));
  CU(ds.alloc(nb_s, s));
  CU(dte.alloc(sizeof(double) * (size_t)opts->n_eval, s));
  CU(dsnap.alloc(nb_snap, s));
  CU(dq.alloc(2 * sizeof(int32_t), s));     // [1]: queue of the team launch (opts->quantum, Radau)
  CU(dst.alloc(nb_stats, s));
  CU(dw.alloc(nb_work, s));
  CU(cudaMemcpyAsync(dy.p, y, nb_y, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dp.p, params, nb_p, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(ds.p, state, nb_s, cudaMemcpyHostToDevice, s));
  if (opts->n_eval) CU(cudaMemcpyAsync(dte.p, t_eval, sizeof(double) * (size_t)opts->n_eval, cudaMemcpyHostToDevice, s));
  if (snapshots && nb_snap) CU(cudaMemcpyAsync(dsnap.p, snapshots, nb_snap, cudaMemcpyHostToDevice, s));
  CU(cudaMemsetAsync(dq.p, 0, 2 * sizeof(int32_t), s));
  CU(cudaMemcpyAsync(dst.p, stats, nb_stats, cudaMemcpyHostToDevice, s));
  rc = implicit_integrate_dev(kind, dy.as<double>(), dp.as<marlpde_column_params>(), ds.as<marlpde_column_state>(),
                              n_columns, n_cells, opts, dte.as<double>(), dsnap.as<double>(), dec.as<int32_t>(),
                              det.as<double>(), dst.as<int64_t>(), dw.p, nb_work, dq.as<int32_t>(), s);
  if (rc) return rc;
  CU(cudaMemcpyAsync(y, dy.p, nb_y, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(state, ds.p, nb_s, cudaMemcpyDeviceToHost, s));
  if (snapshots && nb_snap) CU(cudaMemcpyAsync(snapshots, dsnap.p, nb_snap, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(stats, dst.p, nb_stats, cudaMemcpyDeviceToHost, s));
  if (event_counts) CU(cudaMemcpyAsync(event_counts, dec.p, nb_ec, cudaMemcpyDeviceToHost, s));
  if (event_times && nb_et) CU(cudaMemcpyAsync(event_times, det.p, nb_et, cudaMemcpyDeviceToHost, s));
  if (sync) CU(cudaStreamSynchronize(s));
  return MARLPDE_OK;
}

int marlpde_radau_integrate(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                            int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* t_eval,
                            double* snapshots, int32_t* event_counts, double* event_times, int64_t* stats,
                            int device) {
  return implicit_integrate_host(kRadau, y, params, state, n_columns, n_cells, opts, t_eval, snapshots, event_counts,
                                 event_times, stats, device, cudaStreamPerThread, true);
}

int marlpde_radau_integrate_async(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                                  int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* t_eval,
                                  double* snapshots, int32_t* event_counts, double* event_times, int64_t* stats,
                                  int device, void* stream) {
  return implicit_integrate_host(kRadau, y, params, state, n_columns, n_cells, opts, t_eval, snapshots, event_counts,
                                 event_times, stats, device, (cudaStream_t)stream, false);
}

int marlpde_bdf_integrate(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                          int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* t_eval,
                          double* snapshots, int32_t* event_counts, double* event_times, int64_t* stats, int device) {
  return implicit_integrate_host(kBdf, y, params, state, n_columns, n_cells, opts, t_eval, snapshots, event_counts,
                                 event_times, stats, device, cudaStreamPerThread, true);
}

int marlpde_bdf_integrate_async(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                                int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* t_eval,
                                double* snapshots, int32_t* event_counts, double* event_times, int64_t* stats,
                                int device, void* stream) {
  return implicit_integrate_host(kBdf, y, params, state, n_columns, n_cells, opts, t_eval, snapshots, event_counts,
                                 event_times, stats, device, (cudaStream_t)stream, false);
}

// ---- explicit Runge-Kutta integrators (RK23, DOP853): the implicit integrators' buffers and checks, no statistics ----
static const char* erk_name(marlpde::ErkMethod m) { return m == marlpde::kErkRK23 ? "rk23" : "dop853"; }

static int check_erk_args(marlpde::ErkMethod m, int n_columns, int n_cells, const marlpde_rk45_options* opts) {
  if (!opts) return fail(MARLPDE_EINVAL, "opts is NULL");
  if (n_columns < 0) return fail(MARLPDE_EINVAL, "n_columns < 0");
  if (n_cells < 3) return fail(MARLPDE_EINVAL, "the %s integrator needs n_cells >= 3 (got %d)", erk_name(m), n_cells);
  if (!(opts->rtol > 0.0) || !(opts->atol >= 0.0)) return fail(MARLPDE_EINVAL, "need rtol > 0, atol >= 0");
  if (!(opts->max_step > 0.0)) return fail(MARLPDE_EINVAL, "max_step must be positive (use +inf for none)");
  if (opts->n_eval < 0 || opts->event_capacity < 0) return fail(MARLPDE_EINVAL, "negative n_eval/event_capacity");
  if (opts->quantum != 0) return fail(MARLPDE_EUNSUPPORTED, "opts->quantum is not used by the %s integrator (pass 0)", erk_name(m));
  return MARLPDE_OK;
}

static int erk_integrate_dev(marlpde::ErkMethod m, double* d_y, const marlpde_column_params* d_params,
                             marlpde_column_state* d_state, int n_columns, int n_cells, const marlpde_rk45_options* opts,
                             const double* d_t_eval, double* d_snapshots, int32_t* d_event_counts, double* d_event_times,
                             void* d_workspace, size_t workspace_bytes, int32_t* d_queue, void* stream) {
  int rc = check_erk_args(m, n_columns, n_cells, opts);
  if (rc) return rc;
  if (n_columns == 0) return MARLPDE_OK;
  if (!d_y || !d_params || !d_state || !d_queue || !d_workspace) return fail(MARLPDE_EINVAL, "NULL device pointer");
  if (opts->n_eval > 0 && (!d_t_eval || !d_snapshots)) return fail(MARLPDE_EINVAL, "n_eval > 0 needs t_eval and snapshots");
  if (opts->flags & MARLPDE_FLAG_EVENTS) {
    if (!d_event_counts) return fail(MARLPDE_EINVAL, "MARLPDE_FLAG_EVENTS needs event_counts");
    if (opts->event_capacity > 0 && !d_event_times) return fail(MARLPDE_EINVAL, "event_capacity > 0 needs event_times");
  }
  const size_t need = marlpde::erk_workspace_bytes(m, n_columns, n_cells);
  if (workspace_bytes < need) return fail(MARLPDE_EINVAL, "workspace too small: %zu < %zu bytes", workspace_bytes, need);
  DevProps props;
  rc = current_props(props);
  if (rc) return rc;
  cudaError_t e = marlpde::launch_erk(m, d_y, d_params, d_state, n_columns, n_cells, *opts, d_t_eval, d_snapshots,
                                      d_event_counts, d_event_times, static_cast<double*>(d_workspace), d_queue,
                                      props.sm_count, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, m == marlpde::kErkRK23 ? "rk23 launch" : "dop853 launch");
  return MARLPDE_OK;
}

static int erk_integrate_host(marlpde::ErkMethod m, double* y, const marlpde_column_params* params,
                              marlpde_column_state* state, int n_columns, int n_cells, const marlpde_rk45_options* opts,
                              const double* t_eval, double* snapshots, int32_t* event_counts, double* event_times,
                              int device, cudaStream_t s, bool sync) {
  int rc = check_erk_args(m, n_columns, n_cells, opts);
  if (rc) return rc;
  if (n_columns == 0) return MARLPDE_OK;
  if (!y || !params || !state) return fail(MARLPDE_EINVAL, "NULL pointer");
  if (opts->n_eval > 0 && (!t_eval || !snapshots)) return fail(MARLPDE_EINVAL, "n_eval > 0 needs t_eval and snapshots");
  DeviceScope scope;
  rc = scope.enter(device);
  if (rc) return rc;
  const size_t nb_y = sizeof(double) * 5 * (size_t)n_cells * n_columns;
  const size_t nb_snap = nb_y * (size_t)opts->n_eval;
  const size_t nb_p = sizeof(marlpde_column_params) * (size_t)n_columns;
  const size_t nb_s = sizeof(marlpde_column_state) * (size_t)n_columns;
  const size_t nb_work = marlpde::erk_workspace_bytes(m, n_columns, n_cells);
  const size_t nb_ec = sizeof(int32_t) * MARLPDE_NEVENTS * (size_t)n_columns;
  const size_t nb_et = sizeof(double) * MARLPDE_NEVENTS * (size_t)opts->event_capacity * n_columns;
  DevBuf dy, dp, ds, dte, dsnap, dq, dw, dec, det;
  CU(dy.alloc(nb_y, s));
  CU(dp.alloc(nb_p, s));
  CU(ds.alloc(nb_s, s));
  CU(dte.alloc(sizeof(double) * (size_t)opts->n_eval, s));
  CU(dsnap.alloc(nb_snap, s));
  CU(dq.alloc(sizeof(int32_t), s));
  CU(dw.alloc(nb_work, s));
  CU(dec.alloc(nb_ec, s));
  CU(det.alloc(nb_et, s));
  CU(cudaMemcpyAsync(dy.p, y, nb_y, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dp.p, params, nb_p, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(ds.p, state, nb_s, cudaMemcpyHostToDevice, s));
  if (opts->n_eval) CU(cudaMemcpyAsync(dte.p, t_eval, sizeof(double) * (size_t)opts->n_eval, cudaMemcpyHostToDevice, s));
  if (snapshots && nb_snap) CU(cudaMemcpyAsync(dsnap.p, snapshots, nb_snap, cudaMemcpyHostToDevice, s));
  CU(cudaMemsetAsync(dq.p, 0, sizeof(int32_t), s));
  if (event_counts) CU(cudaMemcpyAsync(dec.p, event_counts, nb_ec, cudaMemcpyHostToDevice, s));
  else CU(cudaMemsetAsync(dec.p, 0, nb_ec, s));
  if (event_times && nb_et) CU(cudaMemcpyAsync(det.p, event_times, nb_et, cudaMemcpyHostToDevice, s));
  marlpde_rk45_options o = *opts;
  o.flags |= model_flags_of(params, n_columns);
  rc = erk_integrate_dev(m, dy.as<double>(), dp.as<marlpde_column_params>(), ds.as<marlpde_column_state>(), n_columns,
                         n_cells, &o, dte.as<double>(), dsnap.as<double>(), dec.as<int32_t>(), det.as<double>(), dw.p,
                         nb_work, dq.as<int32_t>(), s);
  if (rc) return rc;
  CU(cudaMemcpyAsync(y, dy.p, nb_y, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(state, ds.p, nb_s, cudaMemcpyDeviceToHost, s));
  if (snapshots && nb_snap) CU(cudaMemcpyAsync(snapshots, dsnap.p, nb_snap, cudaMemcpyDeviceToHost, s));
  if (event_counts) CU(cudaMemcpyAsync(event_counts, dec.p, nb_ec, cudaMemcpyDeviceToHost, s));
  if (event_times && nb_et) CU(cudaMemcpyAsync(event_times, det.p, nb_et, cudaMemcpyDeviceToHost, s));
  if (sync) CU(cudaStreamSynchronize(s));
  return MARLPDE_OK;
}

size_t marlpde_rk23_workspace_bytes(int n_columns, int n_cells) {
  if (n_columns <= 0 || n_cells <= 0) return 0;
  return marlpde::erk_workspace_bytes(marlpde::kErkRK23, n_columns, n_cells);
}

size_t marlpde_dop853_workspace_bytes(int n_columns, int n_cells) {
  if (n_columns <= 0 || n_cells <= 0) return 0;
  return marlpde::erk_workspace_bytes(marlpde::kErkDOP853, n_columns, n_cells);
}

int marlpde_rk23_integrate_dev(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                               int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* d_t_eval,
                               double* d_snapshots, int32_t* d_event_counts, double* d_event_times, void* d_workspace,
                               size_t workspace_bytes, int32_t* d_queue, void* stream) {
  return erk_integrate_dev(marlpde::kErkRK23, d_y, d_params, d_state, n_columns, n_cells, opts, d_t_eval, d_snapshots,
                           d_event_counts, d_event_times, d_workspace, workspace_bytes, d_queue, stream);
}

int marlpde_dop853_integrate_dev(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                                 int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* d_t_eval,
                                 double* d_snapshots, int32_t* d_event_counts, double* d_event_times, void* d_workspace,
                                 size_t workspace_bytes, int32_t* d_queue, void* stream) {
  return erk_integrate_dev(marlpde::kErkDOP853, d_y, d_params, d_state, n_columns, n_cells, opts, d_t_eval, d_snapshots,
                           d_event_counts, d_event_times, d_workspace, workspace_bytes, d_queue, stream);
}

int marlpde_rk23_integrate(double* y, const marlpde_column_params* params, marlpde_column_state* state, int n_columns,
                           int n_cells, const marlpde_rk45_options* opts, const double* t_eval, double* snapshots,
                           int32_t* event_counts, double* event_times, int device) {
  return erk_integrate_host(marlpde::kErkRK23, y, params, state, n_columns, n_cells, opts, t_eval, snapshots,
                            event_counts, event_times, device, cudaStreamPerThread, true);
}

int marlpde_dop853_integrate(double* y, const marlpde_column_params* params, marlpde_column_state* state, int n_columns,
                             int n_cells, const marlpde_rk45_options* opts, const double* t_eval, double* snapshots,
                             int32_t* event_counts, double* event_times, int device) {
  return erk_integrate_host(marlpde::kErkDOP853, y, params, state, n_columns, n_cells, opts, t_eval, snapshots,
                            event_counts, event_times, device, cudaStreamPerThread, true);
}

int marlpde_rk23_integrate_async(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                                 int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* t_eval,
                                 double* snapshots, int32_t* event_counts, double* event_times, int device,
                                 void* stream) {
  return erk_integrate_host(marlpde::kErkRK23, y, params, state, n_columns, n_cells, opts, t_eval, snapshots,
                            event_counts, event_times, device, (cudaStream_t)stream, false);
}

int marlpde_dop853_integrate_async(double* y, const marlpde_column_params* params, marlpde_column_state* state,
                                   int n_columns, int n_cells, const marlpde_rk45_options* opts, const double* t_eval,
                                   double* snapshots, int32_t* event_counts, double* event_times, int device,
                                   void* stream) {
  return erk_integrate_host(marlpde::kErkDOP853, y, params, state, n_columns, n_cells, opts, t_eval, snapshots,
                            event_counts, event_times, device, (cudaStream_t)stream, false);
}

}  // extern "C"
