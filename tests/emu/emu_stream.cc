// tests/emu/emu_stream.cc — the large-depth-grid RK45 path (csrc/rk45_streaming.cu: init / K1 / tile_attempt / prepare /
// copyback / finish kernels), compiled for the host; its own launcher runs unchanged, every launch executed block by
// block by the SIMT emulator.  TEST INFRASTRUCTURE ONLY (simt_emu.h).
#include <cstdint>
#include <vector>

#include "cuda_runtime.h"
#include "simt_emu.h"

#include "../../integrating-diagenetic-equations-using-python_b200/csrc/rk45_streaming.cu"

extern "C" int emu_rk45_stream(double* y, const marlpde_column_params* params, marlpde_column_state* state, int n_columns,
                               int n_cells, const marlpde_rk45_options* opt, const double* t_eval, double* snap,
                               long long attempts, int32_t* ev_counts, double* ev_times) {
  std::vector<unsigned char> work(marlpde::rk45_stream_workspace_bytes(n_columns, n_cells) + 256, 0);
  return (int)marlpde::launch_rk45_stream(y, params, state, n_columns, n_cells, *opt, t_eval, snap, ev_counts, ev_times, work.data(),
                                          attempts, nullptr);
}
