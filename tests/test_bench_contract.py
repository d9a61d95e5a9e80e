"""bench.py contract on CPU: the reference arm (`--impl reference`) runs the oracle port of the reference's
own path (SciPy RK45 + numba RHS, events on) on the host cores and prints ONE JSON line with the keys the
driver reads; workload descriptions are consistent across world sizes.  (The GPU arm is exercised on the
B200 box by the driver; it needs a CUDA device.)"""
import json
import os
import subprocess
import sys

from conftest import ROOT


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-t-end", "2e-4"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "column RK-steps/sec at N=200" and d["unit"] == "column-steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1 and d["dtype"] == "f64"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == (os.cpu_count() or 1)
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "4096-column" in d["config"]["workload"] and d["config"]["n_cells"] == 200


def test_workload_descriptions_per_world_size():
    sys.path.insert(0, ROOT)
    import bench
    from types import SimpleNamespace
    args = SimpleNamespace(base="default", attempts=3000)
    for world, cols in ((1, 4096), (2, 16384), (4, 32768), (8, 65536)):
        cfg = bench.workload_config(args, world)
        assert cfg["columns"] == cols and cfg["columns_per_gpu"] == cols // world and f"{cols}-column" in cfg["workload"]
    assert bench.lattice_for(1) == (16, 16, 16) and bench.lattice_for(8) == (32, 32, 64)
    assert bench.FLOP_PER_COLUMN_STEP_PER_CELL * 200 == 307600


class _HostStepper:
    """The attributes of bench.Rk45Stepper that dump_outputs reads, on host tensors."""

    def __init__(self, B, N, evcap, counts):
        import numpy as np
        import torch
        from marlpde_b200 import _cabi
        self.B, self.N, self.evcap = B, N, evcap
        self.d_y = torch.arange(B * 5 * N, dtype=torch.float64).reshape(B, 5, N)
        self.d_ec = torch.from_numpy(counts.astype(np.int32))
        et = np.full((B, 7, evcap), np.nan)
        for c, k in np.ndindex(B, 7):                    # the kernel fills slots 0 .. min(count, evcap) - 1
            n = min(int(counts[c, k]), evcap)
            et[c, k, :n] = 1e-3 * (100 * c + 10 * k + np.arange(n))
        self.d_et = torch.from_numpy(et)
        self._st = np.zeros(B, _cabi.STATE_DTYPE)
        self._st["t"], self._st["status"] = 0.5, -1

    def state(self):
        return self._st


def test_dump_outputs_are_finite_float64_and_within_budget(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    counts = np.zeros((4, 7), dtype=np.int64)
    counts[0, 2], counts[3, 0], counts[3, 6] = 1, 3, 20           # 20 > evcap: only the first 16 roots are stored
    bench.dump_outputs(str(tmp_path / "one"), _HostStepper(4, 200, 16, counts), 0, 1)
    got = {p.stem: np.load(p) for p in (tmp_path / "one").iterdir()}
    assert set(got) == {"column_index", "y", "event_counts", "event_times", "state_t", "state_h_abs",
                        "state_n_accepted", "state_n_rejected", "state_nfev", "state_status"}
    for name, a in got.items():
        assert a.dtype == np.float64 and np.all(np.isfinite(a)), name
    assert np.array_equal(got["event_counts"], counts) and got["y"].shape == (4, 5, 200)
    want = [0.02] + [0.3, 0.301, 0.302] + [0.36 + 1e-3 * i for i in range(16)]
    assert np.allclose(got["event_times"], want, rtol=0, atol=1e-12)
    # two ranks of 8192 columns do not fit the budget together: a seeded sample per rank, identical from run to run
    big = np.zeros((8192, 7), dtype=np.int64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), _HostStepper(8192, 200, 16, big), 1, 2)
    sizes = sum(p.stat().st_size for p in (tmp_path / "a").iterdir())
    assert 2 * sizes <= bench.DUMP_BUDGET_BYTES
    for p in (tmp_path / "a").iterdir():
        assert p.name.endswith("_rank1.npy") and np.array_equal(np.load(p), np.load(tmp_path / "b" / p.name))
