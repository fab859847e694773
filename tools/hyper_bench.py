"""
Cost of the batched hyper-parameter gradients (vgpa_hyper_device) next to one F + gradient evaluation
(vgpa_eval_device, want_grad = 1) on the same handle, the same x and the same stream.

    python tools/hyper_bench.py [--reps 5] [--warmup 2] [--only l96|ou|l63]

Workloads:
  l96  bench.py's flagship shard: Lorenz-96 D = 40, N = 1001, RK2, 4096 problems, x = x0 (1 + 0.02 u) generated in HBM
  ou   OU x 1024, RK4, N = 1001 (bench.py secondary configs[1]), x from the on-device initialisation
  l63  L63 x 4096, RK2, N = 2002 (bench.py secondary configs[2]), x from the on-device initialisation
The two calls alternate (hyper, eval, hyper, eval, ...), each timed with CUDA events; the medians are reported
with the per-kind times of vgpa_set_timing (fwd / energy / finalize / bwd, milliseconds per call) from a separate,
untimed pass.  Prints one JSON line with the card's name and power limit.
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def l96_workload(torch, dev):
    from vgpa_b200.engine import BatchEvaluator
    B = bench.PER_GPU
    fam = bench.l96_problem_family(0)
    iset, arr = bench.shard_arrays(fam, B)
    ev = BatchEvaluator("L96", "rk2", bench.N_GRID, bench.DT, [8.0], arr["sigma"], np.ones(bench.D), fam["obs_t"],
                        arr["obs_y"], arr["m0"], fam["s0"], arr["E0"], B=B, dt_model=fam["dt_model"], device=dev.index)
    X = torch.empty((B, bench.N_X), dtype=torch.float64, device=dev)
    x0s = torch.from_numpy(np.stack([s_["x0"] for s_ in fam["sets"]])).to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(bench.SEED % (2 ** 31))
    for p0 in range(0, B, 128):
        p1 = min(B, p0 + 128)
        u = torch.rand((p1 - p0, bench.N_X), dtype=torch.float64, device=dev, generator=gen) * 2.0 - 1.0
        X[p0:p1] = x0s[torch.from_numpy(iset[p0:p1]).to(dev)] * (1.0 + 0.02 * u)
    return ev, X


def small_workload(torch, dev, model, method, tf, sys_noise, obs_noise, density, theta, B):
    """bench.py's secondary batches: one sample path, per-problem observation noise and m0."""
    from vgpa_b200 import Simulation
    from vgpa_b200.engine import BatchEvaluator
    params = {"Output_Name": "bench", "Model": model, "Ode-method": method, "Random-Seed": bench.SEED,
              "Time-window": {"t0": 0.0, "tf": tf, "dt": 0.01}, "Noise": {"sys": sys_noise, "obs": obs_noise},
              "Observations": {"density": density, "operator": None}, "Drift": {"theta": theta},
              "Prior": {"tau0": 0.5, "mu0": 1.0}}
    sim = Simulation("bench")
    sim.setup(params)
    md = sim.m_data
    mdl = md["model"]
    path = np.asarray(mdl.sample_path, dtype=float)
    Dm = 1 if path.ndim == 1 else path.shape[1]
    Nn = path.shape[0]
    obs_t = np.asarray(md["obs_t"], dtype=np.int64)
    R = np.asarray(md["obs_noise"], dtype=float)
    R = np.diagonal(R).copy() if R.ndim == 2 else np.full(Dm, float(R))
    obs_y, m0 = np.empty((B, obs_t.size, Dm)), np.empty((B, Dm))
    for p_ in range(B):
        rng = np.random.default_rng(np.random.SeedSequence([bench.SEED, p_]))
        obs_y[p_] = path.reshape(Nn, Dm)[obs_t] + np.sqrt(R) * rng.standard_normal((Dm, obs_t.size)).T
        m0[p_] = path.reshape(Nn, Dm)[0] + 0.1 * rng.standard_normal(Dm)
    s0 = np.atleast_2d(np.asarray(md["s0"], dtype=float))
    kl0 = sim.build().kl0
    E0 = np.array([float(np.asarray(kl0(m0[p_] if Dm > 1 else m0[p_, 0], md["s0"]))) for p_ in range(B)])
    sigma = np.atleast_1d(np.asarray(mdl.sigma, dtype=float))
    sigma = np.diag(sigma).copy() if sigma.ndim == 2 else sigma
    ev = BatchEvaluator(model, method.lower(), Nn, 0.01, np.atleast_1d(np.asarray(mdl.theta, dtype=float)), sigma, R,
                        obs_t, obs_y, m0, s0, E0, B=B, dt_model=float(mdl.time_step), device=dev.index)
    X = torch.empty((B, ev.n_x), dtype=torch.float64, device=dev)
    ev.initialization_device(X.data_ptr(), ev.n_x, 0.0, torch.cuda.current_stream(dev).cuda_stream)
    ev.sync()
    return ev, X


def measure(torch, ev, X, reps, warmup):
    B, n, D, nth = ev.B, ev.n_x, ev.D, ev.n_theta
    dev = X.device
    st = torch.cuda.current_stream(dev).cuda_stream
    F, Fh, Es = (torch.empty(B, dtype=torch.float64, device=dev) for _ in range(3))
    G = torch.empty_like(X)
    dth = torch.empty((B, nth), dtype=torch.float64, device=dev)
    dsig = torch.empty((B, 1 if D == 1 else D * D), dtype=torch.float64, device=dev)

    def hyper():
        ev.hyper_device(X.data_ptr(), n, Fh.data_ptr(), Es.data_ptr(), dth.data_ptr(), nth, dsig.data_ptr(),
                        dsig.shape[1], st)

    def evaluate():
        ev.eval_device(X.data_ptr(), n, F.data_ptr(), G.data_ptr(), n, st)

    for _ in range(warmup):
        hyper()
        evaluate()
    ev.sync()
    times = {"hyper": [], "eval": []}
    for _ in range(reps):
        for name, fn in (("hyper", hyper), ("eval", evaluate)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            ev.sync()
            times[name].append(e0.elapsed_time(e1))
    assert bool(torch.equal(F, Fh)), "hyper_device F differs from eval_device F"
    assert bool(torch.isfinite(dth).all()) and bool(torch.isfinite(dsig).all())
    kinds = {}
    for name, fn in (("hyper", hyper), ("eval", evaluate)):   # per-kind device time, one untimed call each
        ev.get_timing()
        ev.set_timing(True)
        fn()
        ev.sync()
        kinds[name] = {k: round(v[0], 3) for k, v in ev.get_timing().items() if v[1]}
        ev.set_timing(False)
    med = {k: statistics.median(v) for k, v in times.items()}
    return {"problems": B, "N": ev.N, "method": ev.method,
            "hyper_ms": round(med["hyper"], 3), "eval_F_grad_ms": round(med["eval"], 3),
            "hyper_over_eval": round(med["hyper"] / med["eval"], 4),
            "spread": {k: round((max(v) - min(v)) / statistics.median(v), 4) for k, v in times.items()},
            "kind_ms": kinds}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", choices=["l96", "ou", "l63"], default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("tools/hyper_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    makers = {
        "l96": lambda: l96_workload(torch, dev),
        "ou": lambda: small_workload(torch, dev, "OU", "RK4", 10.0, 0.8, 0.04, 2, 2.0, 1024),
        "l63": lambda: small_workload(torch, dev, "L63", "RK2", 20.0, [10.0] * 3, 2.0, 5, [10.0, 28.0, 2.6667], 4096),
    }
    names = {"l96": "L96_x4096_rk2_N1001", "ou": "OU_x1024_rk4_N1001", "l63": "L63_x4096_rk2_N2002"}
    out = {"gpu": gpu_info(), "reps": args.reps, "timer": "CUDA events around each call, medians"}
    for key, make in makers.items():
        if args.only and key != args.only:
            continue
        ev, X = make()
        with ev:
            out[names[key]] = measure(torch, ev, X, args.reps, args.warmup)
        del X
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
