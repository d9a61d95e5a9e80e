// Host-side declarations of the explicit Runge-Kutta integrators' launcher (RK23, DOP853; internal to the library).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

#include "../../include/marlpde_b200.h"

namespace marlpde {

enum ErkMethod { kErkRK23 = 0, kErkDOP853 = 1 };

size_t erk_workspace_bytes(ErkMethod method, int n_columns, int n_cells);

cudaError_t launch_erk(ErkMethod method, double* d_y, const marlpde_column_params* d_params,
                       marlpde_column_state* d_state, int n_columns, int n_cells, const marlpde_rk45_options& opt,
                       const double* d_t_eval, double* d_snap, int32_t* d_ev_counts, double* d_ev_times,
                       double* d_work, int32_t* d_queue, int sm_count, cudaStream_t stream);

}  // namespace marlpde
