"""Short streaming-RK45 run for ncu: B columns of N cells, a few step attempts per call.
    python scripts/profile_stream.py [N] [B] [attempts]"""
import os, sys, time, ctypes as C
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "integrating-diagenetic-equations-using-python_b200"))
import numpy as np, torch
import marlpde_b200 as mb
from marlpde_b200 import _cabi, batch
from marlpde.parameters import Map_Scenario
from dataclasses import asdict
N = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
B = int(sys.argv[2]) if len(sys.argv) > 2 else 64
att = int(sys.argv[3]) if len(sys.argv) > 3 else 24
pde = asdict(Map_Scenario()) | {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6, "N": N}
P = np.repeat(mb.derive_column_params(pde), B)
y = torch.from_numpy(np.repeat(mb.initial_state(pde), B, 0)).cuda()
dP = batch.params_to_device(P, y.device)
st = torch.from_numpy(batch.make_state(B, 0.0, 1e-6 * (200 / N) ** 2).view(np.uint8).copy()).cuda()
lib = _cabi.lib()
nb = int(lib.marlpde_rk45_stream_workspace_bytes(B, N))
w = torch.empty(nb // 8 + 1, dtype=torch.float64, device="cuda")
o = _cabi.RK45Options(t_bound=1.0, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=att, n_eval=0, event_capacity=0, flags=0, quantum=0)
stream = torch.cuda.current_stream().cuda_stream
for i in range(3):
    torch.cuda.synchronize(); t0 = time.time()
    _cabi.check(lib.marlpde_rk45_stream_integrate_dev(y.data_ptr(), dP.data_ptr(), st.data_ptr(), B, N, C.byref(o), None, None, w.data_ptr(), nb, stream))
    torch.cuda.synchronize(); dt = time.time() - t0
    print(f"call {i}: {att} attempts x {B} columns x {N} cells in {dt*1e3:.2f} ms -> {160.0*N*B*att/dt/1e9:.0f} GB/s algorithmic, {B*att/dt:.3e} column-steps/s")
