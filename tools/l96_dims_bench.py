"""
F + gradient evaluations per second of Lorenz 96 at several state dimensions D (N = 1001, RK2): the run-time-D
kernels (l96_dyn.cu) at D != 40 and the tuned D = 40 kernels in the same run, for scale.

    python tools/l96_dims_bench.py [--dims 10,20,32,40,48,64] [--batch 4096] [--reps 3]

Each D runs at B = 1 and at a batch that fills the GPU (capped so that x and the gradient of the batch fit in
--mem-gb of device memory; the B used is reported).  Every problem has its own x; one untimed evaluation warms up.
The time is the median of --reps device-synchronised evaluations.  A second, untimed-by-the-clock pass reports
the per-kind kernel milliseconds of vgpa_set_timing (0 forward, 1 energy, 2 finalize, 3 backward).  Prints one
JSON line with the card's name and power limit.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def problem_set(D, N, B, dt=0.01, seed=0):
    rng = np.random.default_rng([seed, D])
    obs_t = np.arange(10, N - 1, 10, dtype=np.int64)
    M = obs_t.size
    kw = dict(theta=8.0, sigma=np.ones(D), R=0.5 * np.ones(D), obs_t=obs_t,
              obs_y=rng.standard_normal((B, M, D)), m0=rng.standard_normal(D), s0=(0.2 * np.eye(D)).ravel(), E0=0.0)
    return kw


def run_one(D, N, B, reps, torch):
    from vgpa_b200.engine import BatchEvaluator
    kw = problem_set(D, N, B)
    with BatchEvaluator("L96", "rk2", N, 0.01, B=B, dt_model=0.01, D=D, **kw) as ev:
        n = ev.n_x
        X = torch.empty((B, n), dtype=torch.float64, device="cuda")
        ev.initialization_device(X.data_ptr(), n, 0.0)
        torch.cuda.synchronize()
        X.mul_(1.0 + 0.01 * torch.randn_like(X))
        F = torch.empty(B, dtype=torch.float64, device="cuda")
        G = torch.empty((B, n), dtype=torch.float64, device="cuda")
        ev.eval_device(X.data_ptr(), n, F.data_ptr(), G.data_ptr(), n)
        ev.sync()
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev.eval_device(X.data_ptr(), n, F.data_ptr(), G.data_ptr(), n)
            ev.sync()
            ts.append(time.perf_counter() - t0)
        ev.set_timing(True)
        ev.eval_device(X.data_ptr(), n, F.data_ptr(), G.data_ptr(), n)
        ev.sync()
        ms = [v[0] for v in ev.get_timing().values()]
        ev.set_timing(False)
        ok = bool(torch.isfinite(F).all().item())
        del X, G, F
        torch.cuda.empty_cache()
    t = float(np.median(ts))
    return {"D": D, "B": B, "seconds": round(t, 5), "evals_per_s": round(B / t, 2),
            "us_per_problem_step": round(1e6 * t / (B * N), 4),
            "kernel_ms": [round(float(v), 3) for v in ms], "finite": ok}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dims", default="10,20,32,40,48,64")
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--N", type=int, default=1001)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--mem-gb", type=float, default=60.0)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("l96_dims_bench: no CUDA device")
    out = {"card": card(), "N": a.N, "method": "rk2", "runs": []}
    for D in (int(v) for v in a.dims.split(",")):
        nx = a.N * D * (D + 1)
        cap = max(1, int(a.mem_gb * 2 ** 30 // (2 * 8 * nx)))
        for B in (1, min(a.batch, cap)):
            r = run_one(D, a.N, B, a.reps, torch)
            r["kernels"] = "tuned D = 40" if D == 40 else "run-time D"
            out["runs"].append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
