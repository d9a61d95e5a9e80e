// tests/emu/emu_erk.cc — the batched explicit Runge-Kutta kernel (csrc/erk_batch.cu: RK23, DOP853), compiled for the
// host and run by the SIMT emulator: one CTA of four warps works through all columns of the queue.  TEST INFRASTRUCTURE
// ONLY (simt_emu.h).
#include <cstdint>
#include <vector>

#include "cuda_runtime.h"
#include "simt_emu.h"

#include "../../integrating-diagenetic-equations-using-python_b200/csrc/erk_batch.cu"

// method 0: RK23, 1: DOP853
extern "C" int emu_erk(int method, double* y, const marlpde_column_params* params, marlpde_column_state* state,
                       int n_columns, int n_cells, const marlpde_rk45_options* opt, const double* t_eval, double* snap,
                       int32_t* ev_counts, double* ev_times) {
  using namespace marlpde;
  const ErkMethod m = method == 0 ? kErkRK23 : kErkDOP853;
  std::vector<double> work(erk_workspace_bytes(m, n_columns, n_cells) / sizeof(double) + 16, 0.0);
  int32_t queue = 0;
  imp::Args a;
  a.g_y = y;
  a.g_params = params;
  a.g_state = state;
  a.g_t_eval = t_eval;
  a.g_snap = snap;
  a.g_stats = nullptr;
  a.g_ev_counts = ev_counts;
  a.g_ev_times = ev_times;
  a.g_work = work.data();
  a.g_queue = &queue;
  a.n_columns = n_columns;
  a.N = n_cells;
  a.opt = *opt;
  return simt::run_block(imp::kWarpsPerCta * 32, 0, [&]() {
    const bool vd = (a.opt.flags & MARLPDE_FLAG_VAR_DPHI) != 0;
    if (m == kErkRK23) {
      if (vd) erk::erk_kernel<erk::RK23, true>(a);
      else erk::erk_kernel<erk::RK23, false>(a);
    } else {
      if (vd) erk::erk_kernel<erk::DOP853, true>(a);
      else erk::erk_kernel<erk::DOP853, false>(a);
    }
  });
}
