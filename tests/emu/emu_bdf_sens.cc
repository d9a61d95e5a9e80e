// tests/emu/emu_bdf_sens.cc — the BDF kernel's sensitivity build (csrc/bdf_batch.cu, bdf_kernel<., ., true>), compiled for
// the host and run by the SIMT emulator: one CTA of four warps works through all columns of the queue.
// TEST INFRASTRUCTURE ONLY (simt_emu.h).
#include <cstdint>
#include <vector>

#include "cuda_runtime.h"
#include "simt_emu.h"

#include "../../integrating-diagenetic-equations-using-python_b200/csrc/bdf_batch.cu"

extern "C" int emu_bdf_sens(double* y, const marlpde_column_params* params, marlpde_column_state* state, int n_columns,
                            int n_cells, const marlpde_rk45_options* opt, const double* t_eval, double* snap,
                            int64_t* stats, int32_t* ev_counts, double* ev_times, int n_dirs,
                            const marlpde_column_params* params_pm, const double* inv2sigma, const double* atol_s,
                            double* sens, double* sens_snap, int64_t* sens_stats) {
  using namespace marlpde;
  std::vector<double> work(bd::work_doubles(n_cells) * (size_t)n_columns + 16, 0.0);
  std::vector<double> swork(bd::sens_work_doubles(n_cells, n_dirs) * (size_t)n_columns + 16, 0.0);
  int32_t queue = 0;
  bd::SensArgs a;
  a.g_y = y;
  a.g_params = params;
  a.g_state = state;
  a.g_t_eval = t_eval;
  a.g_snap = snap;
  a.g_stats = stats;
  a.g_ev_counts = ev_counts;
  a.g_ev_times = ev_times;
  a.g_work = work.data();
  a.g_queue = &queue;
  a.n_columns = n_columns;
  a.N = n_cells;
  a.opt = *opt;
  a.g_params_pm = params_pm;
  a.g_inv2sigma = inv2sigma;
  a.g_atol_s = atol_s;
  a.g_sens = sens;
  a.g_sens_snap = sens_snap;
  a.g_sens_stats = sens_stats;
  a.g_sens_work = swork.data();
  a.n_dirs = n_dirs;
  return simt::run_block(imp::kWarpsPerCta * 32, 0, [&]() {
    const bool vd = (a.opt.flags & MARLPDE_FLAG_VAR_DPHI) != 0, fd = (a.opt.flags & MARLPDE_FLAG_JAC_FD) != 0;
    if (vd && fd) bd::bdf_kernel<true, true, true>(a);
    else if (vd) bd::bdf_kernel<true, false, true>(a);
    else if (fd) bd::bdf_kernel<false, true, true>(a);
    else bd::bdf_kernel<false, false, true>(a);
  });
}
