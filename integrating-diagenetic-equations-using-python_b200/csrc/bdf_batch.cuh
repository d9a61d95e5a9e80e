// Host-side declarations of the variable-order BDF integrator's launcher (internal to the library).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

#include "../../include/marlpde_b200.h"

namespace marlpde {

size_t bdf_workspace_bytes(int n_columns, int n_cells);

cudaError_t launch_bdf(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                       int n_columns, int n_cells, const marlpde_rk45_options& opt, const double* d_t_eval,
                       double* d_snap, int64_t* d_stats, int32_t* d_ev_counts, double* d_ev_times, double* d_work,
                       int32_t* d_queue, int sm_count, cudaStream_t stream);

// forward sensitivities (bdf_kernel<., ., true>): see marlpde_bdf_sens_integrate_dev
constexpr int kBdfMaxDirs = 8;
size_t bdf_sens_workspace_bytes(int n_columns, int n_cells, int n_dirs);
cudaError_t launch_bdf_sens_check(const marlpde_column_params* d_params, const marlpde_column_params* d_params_pm,
                                  int n_columns, int n_dirs, int32_t* d_bad, cudaStream_t stream);
cudaError_t launch_bdf_sens(double* d_y, const marlpde_column_params* d_params, marlpde_column_state* d_state,
                            int n_columns, int n_cells, const marlpde_rk45_options& opt, const double* d_t_eval,
                            double* d_snap, int64_t* d_stats, int32_t* d_ev_counts, double* d_ev_times, double* d_work,
                            int32_t* d_queue, int n_dirs, const marlpde_column_params* d_params_pm,
                            const double* d_inv2sigma, const double* d_atol_s, double* d_sens, double* d_sens_snap,
                            int64_t* d_sens_stats, double* d_sens_work, int sm_count, cudaStream_t stream);

}  // namespace marlpde
