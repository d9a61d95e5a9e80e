"""Cost of the BDF integrator's forward sensitivities (csrc/bdf_batch.cu, bdf_kernel<., ., true>) in one GPU call:
the 4096-column lattice (sweep_lattice(default, 16, 16, 16)), N = 200, to t = 0.05, with P = 0, 1, 2, 4 directions
(k2, DCO3, b, and S moved consistently with Xstar and Tstar), device path, each timed with a device synchronise after a
warm-up run of the same shape.  For each P: wall time, ratio to P = 0, and per column the mean sensitivity corrector
iterations, fallback factorisations and unconverged steps; plus the card's name and power limit.

    python scripts/profile_sensitivity.py [t_end] [repeats]
Prints one JSON document."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "integrating-diagenetic-equations-using-python_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import marlpde_b200 as mb  # noqa: E402
from marlpde.parameters import Map_Scenario  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def main():
    t_end = float(sys.argv[1]) if len(sys.argv) > 1 else 0.05
    repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 2
    if not torch.cuda.is_available():
        raise SystemExit("profile_sensitivity.py needs a CUDA device")
    from dataclasses import asdict
    lat = mb.sweep_lattice(asdict(Map_Scenario()), 16, 16, 16)
    S, D0Ca = lat["sedimentationrate"], lat["D0Ca"]
    all_dirs = ["k2", "DCO3", "b", {"sedimentationrate": 1.0, "Xstar": -D0Ca / S ** 2, "Tstar": -2.0 * D0Ca / S ** 3}]
    P = mb.derive_column_params(lat)
    y0 = torch.from_numpy(mb.initial_state(lat)).cuda()
    d_params = mb.batch.params_to_device(P, y0.device)
    out = {"card": card(), "columns": int(P.shape[0]), "n_cells": int(y0.shape[2]), "t_end": t_end, "runs": []}
    base = None
    for nd in (0, 1, 2, 4):
        sd = mb.sensitivity_directions(lat, all_dirs[:nd]) if nd else None
        kw = dict(t_span=(0, t_end), first_step=1e-6, t_eval=[t_end], sensitivities=sd)
        mb.integrate_bdf_batch(y0, d_params, **kw)                    # warm-up (module load, pool)
        torch.cuda.synchronize()
        times = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            r = mb.integrate_bdf_batch(y0, d_params, **kw)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        best = min(times)
        base = best if nd == 0 else base
        row = {"P": nd, "seconds": best, "all_seconds": times, "ratio_to_P0": best / base,
               "finished": int(np.sum(r.status == 0)), "mean_accepted": float(np.mean(r.n_accepted))}
        if nd:
            st = r.sens_stats
            row.update(directions=sd.names, mean_corrector_iterations=float(st[:, 0].mean()),
                       mean_iterations_per_step_and_direction=float(st[:, 0].sum() / max(1, r.n_accepted.sum()) / nd),
                       mean_fallback_factorisations=float(st[:, 1].mean()),
                       mean_unconverged_steps=float(st[:, 2].mean()), columns_with_unconverged=int(np.sum(st[:, 2] > 0)))
        out["runs"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
