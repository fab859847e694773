#!/usr/bin/env python
"""
bench.py -- VGPA free-energy + gradient evaluations per second on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[4], the one the metric is quoted on): the Lorenz-96
D=40, T=1000 (N=1001 grid points, RK2) ensemble of 32768 independent inference
problems = 64 observation sets x 32 starts x 16 system-noise values, sharded as
contiguous blocks of 4096 problems per GPU (weak scaling: per-GPU work is fixed;
8 GPUs = the full 32768).  One "step" = free_energy + gradient for every problem of
the shard, x and grad resident in HBM.  NCCL is used only to gather F.

Besides the contract keys the b200 line carries (N = 1): `cpu_baseline` (the C port of the reference
algorithm on the host cores), `cpu_baseline_reference` (the UNMODIFIED Python reference from
baseline/_ref, one warm evaluation, with a live parity check of the CUDA path against it),
`secondary` (the other BASELINE configs, a few seconds each) and `e2e.copy_ceiling_gbs` (pure pinned
H2D + D2H copies running concurrently: the ceiling the host-buffer API can reach on this box).

JSON keys follow the driver contract; see DESIGN.md section "Measurement".
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SEED = 31415926535
D, N_GRID, M_OBS, DT = 40, 1001, 80, 0.01
N_X = N_GRID * D * (D + 1)
PER_GPU = 4096
N_OBS_SETS_PER_GPU, N_STARTS, N_NOISE = 8, 32, 16
# algorithmic work per (problem, time index), SURVEY.md 8(d)
FLOP_STEP = {"fwd": 262400.0, "energy": 429867.0, "bwd": 262400.0 + 265600.0}
BYTE_STEP = {"fwd": 2 * 8.0 * D * (D + 1), "energy": 3 * 8.0 * D * (D + 1), "bwd": 4 * 8.0 * D * (D + 1)}
FLOP_EVAL = 1.2215e9
BYTE_EVAL = 9 * 8.0 * N_GRID * D * (D + 1)
# FP64 peaks measured on this pool's B200 by tools/microbench.cu (profiles/microbench_r01.jsonl)
FP64_DFMA_TFLOPS, FP64_DMMA_TFLOPS = 33.9, 37.1


def l96_params(tf=10.0):
    return {"Output_Name": "bench", "Model": "L96", "Ode-method": "RK2", "Random-Seed": SEED,
            "Time-window": {"t0": 0.0, "tf": tf, "dt": DT}, "Noise": {"sys": [4.0] * D, "obs": 1.0},
            "Observations": {"density": 8, "operator": None}, "Drift": {"theta": 8.0},
            "Prior": {"tau0": 0.5, "mu0": 1.0}}


def _family_sets(rank, path, obs_t, make_set):
    sets = []
    for s_ in range(N_OBS_SETS_PER_GPU):
        g = rank * N_OBS_SETS_PER_GPU + s_
        rng = np.random.default_rng(np.random.SeedSequence([SEED, g]))
        obs_y = path[obs_t] + rng.standard_normal((obs_t.size, D))          # R = 1
        m0 = path[0] + 0.1 * rng.standard_normal(D)
        sets.append(make_set(obs_y, m0))
    noise = np.array([4.0 * 2.0 ** ((j - 8) / 8.0) for j in range(N_NOISE)])
    return sets, noise


def l96_problem_family(rank):
    """The shard of the C5 ensemble owned by `rank`: 8 observation sets x 32 starts x 16
    noise values.  Host side: one sample path, per-set observations and the reference's
    cubic-spline initialisation (VarGP.initialization) -- identical code to the single
    problem path (vgpa_b200's host mirror of the reference set-up)."""
    from vgpa_b200.simulation import Simulation
    sim = Simulation("bench")
    sim.setup(l96_params())
    md = sim.m_data
    path = md["model"].sample_path
    obs_t = np.asarray(md["obs_t"], dtype=np.int64)

    def make_set(obs_y, m0):
        md["obs_y"], md["m0"] = obs_y, m0
        vg = sim.build()
        return dict(obs_y=obs_y, m0=m0, x0=vg.initialization(), E0=float(vg.kl0(m0, md["s0"])))
    sets, noise = _family_sets(rank, path, obs_t, make_set)
    return dict(obs_t=obs_t, sets=sets, noise=noise, s0=md["s0"], dt_model=float(md["model"].time_step))


def l96_problem_family_cpu(rank=0):
    """The same family WITHOUT importing vgpa_b200 (the CPU arm must not map the CUDA library): the
    set-up comes from the unmodified reference in baseline/_ref when it is importable here (the host
    mirror reproduces it bit for bit), else from numpy + the oracle's make_trajectory; x0 and E0 from
    the oracle's restatements of VarGP.initialization and PriorKL0."""
    from oracle import Oracle, Problem, prior_kl0
    orc = Oracle()
    s0, mu0, tau0 = 0.2 * np.eye(D), np.ones(D), 0.5 * np.eye(D)
    try:
        from baseline.refload import import_reference, reference_objects
        sim, _ = reference_objects(import_reference(), l96_params())
        md = sim.m_data
        path = np.asarray(md["model"].sample_path)
        obs_t = np.asarray(md["obs_t"], dtype=np.int64)
        dt_model = float(md["model"].time_step)
        source = "baseline/_ref"
    except Exception:     # no numba / no reference copy on this box: same shapes, numpy draws
        rng = np.random.default_rng(np.random.SeedSequence(SEED))
        z = rng.standard_normal((D, N_GRID))
        path = orc.make_trajectory("L96", N_GRID, DT, [8.0], np.full(D, 4.0), z)
        obs_t = np.arange(8, N_GRID, 12, dtype=np.int64)[:M_OBS]
        dt_model = DT
        source = "numpy + oracle"

    def make_set(obs_y, m0):
        E0 = float(prior_kl0(m0, s0, mu0, tau0, False))
        prob = Problem(model="L96", method="rk2", D=D, N=N_GRID, dt=DT, theta=np.array([8.0]), sigma=np.full(D, 4.0),
                       R=np.ones(D), obs_t=obs_t, obs_y=obs_y, m0=m0, s0=s0, E0=E0, dt_model=dt_model)
        return dict(obs_y=obs_y, m0=m0, x0=orc.initialization(prob, 0.0), E0=E0)
    sets, noise = _family_sets(rank, path, obs_t, make_set)
    return dict(obs_t=obs_t, sets=sets, noise=noise, s0=s0, dt_model=dt_model, source=source)


def shard_arrays(fam, count):
    """Per-problem parameter arrays for `count` problems of the shard, index
    p = (set * 32 + start) * 16 + noise."""
    idx = np.arange(count)
    iset = idx // (N_STARTS * N_NOISE)
    inoise = idx % N_NOISE
    obs_y = np.stack([fam["sets"][s]["obs_y"] for s in iset])
    m0 = np.stack([fam["sets"][s]["m0"] for s in iset])
    E0 = np.array([fam["sets"][s]["E0"] for s in iset])
    sigma = np.repeat(fam["noise"][inoise][:, None], D, axis=1)
    return iset, dict(obs_y=obs_y, m0=m0, E0=E0, sigma=sigma)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def cpu_port_rate(threads, problems, fam=None):
    """The oracle (C port of the reference algorithm) on the host cores: `problems`
    evaluations of the L96 N=1001 problem, one OpenMP thread per problem."""
    from oracle import Oracle, Problem
    fam = fam or l96_problem_family_cpu(0)
    s = fam["sets"][0]
    orc = Oracle()
    probs = [Problem(model="L96", method="rk2", D=D, N=N_GRID, dt=DT, theta=np.array([8.0]),
                     sigma=np.full(D, 4.0), R=np.ones(D), obs_t=fam["obs_t"], obs_y=s["obs_y"], m0=s["m0"],
                     s0=fam["s0"], E0=s["E0"], dt_model=fam["dt_model"]) for _ in range(problems)]
    rng = np.random.default_rng(5)
    X = np.stack([s["x0"] * (1.0 + 0.02 * rng.uniform(-1, 1, N_X)) for _ in range(problems)])
    t0 = time.perf_counter()
    F, G = orc.eval_batch(probs, X, want_grad=True, threads=threads)
    el = time.perf_counter() - t0
    assert np.all(np.isfinite(F))
    return problems / el, el


def reference_python_rate(override=None):
    """The UNMODIFIED reference (baseline/_ref: numpy / scipy / numba) on this box's CPU: ONE warm
    free_energy(x0) + gradient(x0) of the L96 D=40 N=1001 RK2 problem through the reference's own
    VarGP (src/var_bayes/simulation.py:189-231), after a short-window evaluation that compiles the
    numba kernels.  `override`: dict(obs_y, m0) replacing the simulation's own observation set, so that
    the CUDA path can be checked against this very evaluation.  Returns a cpu_baseline-style dict (with
    F_x0 and the seconds spent), or a dict with `unavailable`."""
    try:
        from baseline.refload import import_reference, reference_objects
        ref = import_reference()
    except Exception as e:
        return {"kind": "reference", "unavailable": f"{type(e).__name__}: {e}"[:200]}
    t_all = time.perf_counter()
    _, args = reference_objects(ref, l96_params(tf=0.3))
    v = ref["VarGP"](*args)
    xs = v.initialization()
    v.free_energy(xs)
    v.gradient(xs)                                   # numba kernels compiled
    _, args = reference_objects(ref, l96_params(), override)
    v = ref["VarGP"](*args)
    x0 = v.initialization()
    t0 = time.perf_counter()
    F = v.free_energy(x0)
    g = v.gradient(x0)
    el = time.perf_counter() - t0
    return {"value": 1.0 / el, "unit": "evals/s", "cores": len(os.sched_getaffinity(0)), "kind": "reference",
            "sample": f"1 warm free_energy + gradient of L96 D=40 N=1001 RK2 through the unmodified reference's VarGP "
                      f"(numpy/numba, one process, default BLAS threads): {el:.1f} s; "
                      f"{time.perf_counter() - t_all:.0f} s including set-up and numba compilation",
            "F_x0": float(F), "gnorm_x0": float(np.linalg.norm(g)), "x0": x0, "grad": g}


def cpu_port_scg_rate(threads, fam):
    """The same ensemble OPTIMISATION on the host cores: one problem per thread, the reference's own SCG
    (baseline/_ref: src/numerics/optim_scg.py) driving the C port's free energy + gradient (one evaluation
    per distinct x, as VarGP's cache gives the CUDA path).  Bounded sample: `threads` problems."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import Oracle, Problem
    try:
        from baseline.refload import import_reference
        SCG = import_reference()["SCG"]
    except Exception as e:
        return {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    orc = Oracle()

    def one(k):
        s_ = fam["sets"][k % len(fam["sets"])]
        prob = Problem(model="L96", method="rk2", D=D, N=N_GRID, dt=DT, theta=np.array([8.0]),
                       sigma=np.full(D, fam["noise"][k % N_NOISE]), R=np.ones(D), obs_t=fam["obs_t"], obs_y=s_["obs_y"],
                       m0=s_["m0"], s0=fam["s0"], E0=s_["E0"], dt_model=fam["dt_model"])
        rng = np.random.default_rng([SEED, 77, k])
        x0 = s_["x0"] * (1.0 + 0.02 * rng.uniform(-1, 1, N_X))
        last = {"x": None}

        def both(x):
            if last["x"] is None or not np.array_equal(x, last["x"]):
                last["F"], last["g"] = orc.eval(prob, x)
                last["x"] = x.copy()
                last["n"] = last.get("n", 0) + 1
            return last
        opt = SCG(lambda x: float(both(x)["F"]), lambda x, eval_fun=False: both(x)["g"].copy(),
                  {"max_it": 500, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False})
        _, fx = opt(x0)
        return int(opt.stats["MaxIt"]), last["n"], float(fx)
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):      # the optimiser's own messages (redirected once, not per thread)
        with ThreadPoolExecutor(max_workers=threads) as ex:
            res = list(ex.map(one, range(threads)))
    el = time.perf_counter() - t0
    return {"optimisations_per_s": threads / el, "problems": threads, "threads": threads, "seconds": el,
            "iterations_median": int(np.median([r[0] for r in res])), "port_evaluations": int(sum(r[1] for r in res)),
            "what": "reference SCG (baseline/_ref) over the C port's evaluation, one problem per host thread"}


METRIC = "free-energy+grad evals/sec (L96 D=40, T=1000); batched problems/sec"
WORKLOAD = ("L96 D=40 N=1001 (T=1000) RK2 ensemble: 8 obs sets x 32 starts x 16 noise values per GPU "
            "(BASELINE configs[4])")


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (the oracle port; the reference is
    Python and cannot travel to the box) on all host cores, same metric/config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = len(os.sched_getaffinity(0))
    fam = l96_problem_family_cpu(0)
    per_step = 4 * max(threads, 1)     # several problems per thread: the step is not paced by one slow thread
    for _ in range(args.warmup):
        cpu_port_rate(threads, min(per_step, 2 * threads), fam)
    n, el = 0, 0.0
    for _ in range(args.steps):
        el += cpu_port_rate(threads, per_step, fam)[1]
        n += per_step
    val = n / el
    line = {"impl": "reference", "metric": METRIC, "value": val,
            "unit": "evals/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * el / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "problems_per_step": per_step},
            "cpu_baseline": {"value": val, "unit": "evals/s", "cores": threads, "kind": "port",
                             "sample": f"{per_step} problems per step on {threads} OpenMP threads (one problem per thread at a time)"},
            "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            # what this arm times: the C / OpenMP restatement of the reference algorithm (oracle/vgpa_oracle.c),
            # NOT the Python reference itself, which is ~400 times slower (calibration below)
            "reference_kind": "port", "problem_family_from": fam.get("source")}
    if args.gpus == 1 and not args.no_python_reference:
        cal = reference_python_rate()
        cal.pop("x0", None)
        cal.pop("grad", None)
        line["cpu_baseline_reference"] = cal
    if args.gpus == 1 and args.scg_problems > 0:
        line["ensemble_scg"] = cpu_port_scg_rate(threads, fam)
    print(json.dumps(line), flush=True)


def copy_ceiling(torch, dist, dev, world, nbytes=1 << 30, reps=3):
    """Pure-copy ceiling of the host-buffer API on this box: one pinned H2D and one pinned D2H
    cudaMemcpyAsync of `nbytes` each, CONCURRENTLY on two streams, on every rank at once (the e2e path
    moves 13 MB in and 13 MB out per evaluation, overlapped).  Returns GB/s per direction, summed over
    the ranks (device-timed, max over ranks)."""
    n = nbytes // 8
    h_in = torch.empty(n, dtype=torch.float64, pin_memory=True)
    h_out = torch.empty(n, dtype=torch.float64, pin_memory=True)
    h_in.fill_(1.0)
    d_in = torch.empty(n, dtype=torch.float64, device=dev)
    d_out = torch.ones(n, dtype=torch.float64, device=dev)
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))

    def once():
        with torch.cuda.stream(s_in):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s_out):
            h_out.copy_(d_out, non_blocking=True)
    once()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    e0.record()
    s_in.wait_event(e0)
    s_out.wait_event(e0)
    for _ in range(reps):
        once()
    e1.record(s_in)
    e2.record(s_out)
    torch.cuda.synchronize()
    ms = max(e0.elapsed_time(e1), e0.elapsed_time(e2))
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    del d_in, d_out, h_in, h_out
    return world * reps * nbytes / (float(t.item()) * 1e-3) / 1e9


def ensemble_scg(torch, dist, dev, local, rank, world, fam, per_gpu):
    """What BASELINE configs[4] describes in full: every member of the ensemble OPTIMISED (SCG to convergence),
    device-resident, sharded over the GPUs -- vgpa_b200.batched_scg.ShardedBatchedSCG on `per_gpu` members
    of each rank's shard (multi-start x noise sweep of the first observation sets), starting points
    x0 * (1 + 0.02 u) generated in HBM.  Whole-job optimisations/s, timed on the host around the sharded
    run (it ends in the NCCL gather), max over ranks."""
    from vgpa_b200.batched_scg import ShardedBatchedSCG
    from vgpa_b200.engine import BatchEvaluator
    iset, arr = shard_arrays(fam, per_gpu)

    def make(lo, hi):
        a, b_ = lo - rank * per_gpu, hi - rank * per_gpu
        return BatchEvaluator("L96", "rk2", N_GRID, DT, [8.0], arr["sigma"][a:b_], np.ones(D), fam["obs_t"],
                              arr["obs_y"][a:b_], arr["m0"][a:b_], fam["s0"], arr["E0"][a:b_], B=b_ - a,
                              dt_model=fam["dt_model"], device=local)

    x0s = torch.from_numpy(np.stack([s_["x0"] for s_ in fam["sets"]])).to(dev)

    def x0_fn(lo, hi, X):
        a = lo - rank * per_gpu
        gen = torch.Generator(device=dev)
        gen.manual_seed(SEED % (2 ** 31) + 1000 + lo)
        for p0 in range(0, hi - lo, 64):
            p1 = min(hi - lo, p0 + 64)
            u = torch.rand((p1 - p0, N_X), dtype=torch.float64, device=dev, generator=gen) * 2.0 - 1.0
            X[p0:p1] = x0s[torch.from_numpy(iset[a + p0:a + p1]).to(dev)] * (1.0 + 0.02 * u)
    # warm-up: two iterations of the first few members of each shard (lazily loaded modules, the first NCCL gather)
    nw = min(per_gpu, 8)
    shift = rank * (per_gpu - nw)            # warm-up problem k of this rank = problem k + shift of the real numbering
    warm = ShardedBatchedSCG(nw * world, lambda lo, hi: make(lo + shift, hi + shift),
                             {"max_it": 2, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}, rank=rank, world=world)
    warm.run(x0_fn=lambda lo, hi, X: x0_fn(lo + shift, hi + shift, X))
    del warm
    ens = ShardedBatchedSCG(per_gpu * world, make, {"max_it": 500, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False},
                            rank=rank, world=world)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    res = ens.run(x0_fn=x0_fn)
    torch.cuda.synchronize()
    print(f"[ensemble_scg] rank {rank}: {time.perf_counter() - t0:.3f} s, phases {res['rank_phase_seconds']}", file=sys.stderr, flush=True)
    el = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    useful = torch.tensor([float(res["f_eval"][rank * per_gpu:(rank + 1) * per_gpu].sum())], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
        dist.all_reduce(useful, op=dist.ReduceOp.SUM)
    el = float(el.item())
    assert np.all(np.isfinite(res["fx"]))
    return {"optimisations_per_s": per_gpu * world / el, "problems": per_gpu * world, "problems_per_gpu": per_gpu,
            "seconds": el, "optimise_seconds_rank0": round(float(res["rank_optimise_seconds"]), 3),
            "phase_seconds_rank0": res["rank_phase_seconds"],
            "iterations_min_median_max": [int(res["n_it"].min()), int(np.median(res["n_it"])), int(res["n_it"].max())],
            "f_evaluations_per_s": float(useful.item()) / el,
            "resident_sub_batch": int(res["sub_batch"]), "device_buffers_per_problem": 5,
            "host_syncs_per_iteration": round(res["rank_host_syncs"] / max(int(res["n_it"][rank * per_gpu:(rank + 1) * per_gpu].max()), 1), 2),
            "fx_mean": float(np.mean(res["fx"])),
            "what": "SCG to convergence (max_it 500, x_tol 1e-6, f_tol 1e-8) of every ensemble member, device-resident; "
                    "f_evaluations counts the reference's f(x) calls (optim_scg.py stats['f_eval']); `seconds` is the whole "
                    "sharded run (evaluator and buffer allocation, starting points, optimisation, gather), "
                    "optimise_seconds_rank0 the optimiser alone"}


def secondary_configs(torch, local, hbm_peak, with_reference=True):
    """The other BASELINE configs, measured in the same run (a few seconds each), each with the bound that
    applies: configs[0] one Double-Well problem through VarGP / SCG (and the unmodified reference beside it),
    configs[1] OU x 1024 RK4 and configs[2] L63 x 4096 RK2 (device-resident batch evaluation, x0
    from the on-device initialisation; HBM bytes 9 * 8 * N * D * (D + 1) per evaluation, SURVEY 8d),
    configs[3] L96 single problem: latency of one free_energy + gradient pair through VarGP (host numpy in
    and out) and the full SCG optimisation to convergence through Simulation / VarGP / SCG."""
    from vgpa_b200 import SCG, Simulation
    from vgpa_b200.engine import BatchEvaluator
    dev = torch.device("cuda", local)
    out = {}

    def base(model, method, tf, sys_noise, obs_noise, density, theta):
        return {"Output_Name": "bench", "Model": model, "Ode-method": method, "Random-Seed": SEED,
                "Time-window": {"t0": 0.0, "tf": tf, "dt": 0.01}, "Noise": {"sys": sys_noise, "obs": obs_noise},
                "Observations": {"density": density, "operator": None}, "Drift": {"theta": theta},
                "Prior": {"tau0": 0.5, "mu0": 1.0}}

    def batch(name, params, Bn, steps=5):
        sim = Simulation("bench")
        sim.setup(params)
        md = sim.m_data
        model = md["model"]
        path = np.asarray(model.sample_path, dtype=float)
        Dm = 1 if path.ndim == 1 else path.shape[1]
        Nn = path.shape[0]
        obs_t = np.asarray(md["obs_t"], dtype=np.int64)
        R = np.asarray(md["obs_noise"], dtype=float)
        R = np.diagonal(R).copy() if R.ndim == 2 else np.full(Dm, float(R))
        obs_y = np.empty((Bn, obs_t.size, Dm))
        m0 = np.empty((Bn, Dm))
        for p_ in range(Bn):                      # SURVEY 8(d): per-problem observation noise and m0
            rng = np.random.default_rng(np.random.SeedSequence([SEED, p_]))
            obs_y[p_] = path.reshape(Nn, Dm)[obs_t] + np.sqrt(R) * rng.standard_normal((Dm, obs_t.size)).T
            m0[p_] = path.reshape(Nn, Dm)[0] + 0.1 * rng.standard_normal(Dm)
        s0 = np.atleast_2d(np.asarray(md["s0"], dtype=float))
        kl0 = sim.build().kl0
        E0 = np.array([float(np.asarray(kl0(m0[p_] if Dm > 1 else m0[p_, 0], md["s0"]))) for p_ in range(Bn)])
        sigma = np.atleast_1d(np.asarray(model.sigma, dtype=float))
        sigma = np.diag(sigma).copy() if sigma.ndim == 2 else sigma
        with BatchEvaluator(params["Model"], params["Ode-method"].lower(), Nn, 0.01,
                            np.atleast_1d(np.asarray(model.theta, dtype=float)), sigma, R, obs_t, obs_y, m0, s0, E0,
                            B=Bn, dt_model=float(model.time_step), device=local) as ev:
            nx = ev.n_x
            X = torch.empty((Bn, nx), dtype=torch.float64, device=dev)
            G = torch.empty_like(X)
            F = torch.empty(Bn, dtype=torch.float64, device=dev)
            st = torch.cuda.current_stream().cuda_stream
            ev.initialization_device(X.data_ptr(), nx, float(params["Time-window"]["t0"]), st)
            for _ in range(3):
                ev.eval_device(X.data_ptr(), nx, F.data_ptr(), G.data_ptr(), nx, st)
            ev.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                ev.eval_device(X.data_ptr(), nx, F.data_ptr(), G.data_ptr(), nx, st)
            e1.record()
            ev.sync()
            ms = e0.elapsed_time(e1) / steps
            assert bool(torch.isfinite(F).all())
        gbs = Bn * 9 * 8.0 * Nn * Dm * (Dm + 1) / (ms * 1e-3) / 1e9
        out[name] = {"problems": Bn, "N": Nn, "method": params["Ode-method"].lower(), "ms_per_batch_eval": round(ms, 4),
                     "evals_per_s": round(Bn / (ms * 1e-3), 1),
                     "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": hbm_peak, "unit": "GB/s",
                                  "frac": round(gbs / hbm_peak, 4)},
                     "l2": ("working set (x + grad) %.0f MB: %s" % (Bn * 2 * 8.0 * nx / 1e6, "larger than the 126 MB L2"
                            if Bn * 2 * 8.0 * nx > 126e6 else "fits the 126 MB L2 (not flushed between iterations: stated)"))}
        if Dm == 1:
            out[name]["note"] = ("one fused time-parallel launch per evaluation (small_dim.cu scan1_eval_kernel): HBM sees x and "
                                 "the gradient only, 2/9 of the three-phase byte count the roofline entry is computed from; "
                                 "the kernel is bound by the FP64 pipe and its barriers, not by HBM")
        del X, G, F

    batch("OU_x1024_rk4_N1001", base("OU", "RK4", 10.0, 0.8, 0.04, 2, 2.0), 1024)
    batch("L63_x4096_rk2_N2002", base("L63", "RK2", 20.0, [10.0] * 3, 2.0, 5, [10.0, 28.0, 2.6667]), 4096)

    # configs[0]: the reference's own CPU case -- one Double-Well problem (sim_params_DW.json: Euler, tf = 10,
    # dt = 0.01), free_energy + gradient pairs and the whole SCG optimisation through Simulation / VarGP / SCG
    # (host numpy in and out), with the unmodified reference timed beside it on this box when it is here
    dw = base("DW", "Euler", 10.0, 0.8, 0.04, 2, 1.0)
    sim = Simulation("bench")
    sim.setup(dw)
    v = sim.build()
    x0 = v.initialization()
    rng = np.random.default_rng(1)
    xs = [x0 * (1.0 + 1e-3 * rng.uniform(-1, 1, x0.size)) for _ in range(4)]
    for x_ in xs:
        v.free_energy(x_)
        v.gradient(x_)
    ts = []
    for i in range(40):
        t0 = time.perf_counter()
        v.free_energy(xs[i % 4])
        v.gradient(xs[i % 4])
        ts.append(time.perf_counter() - t0)
    scg = SCG(v.free_energy, v.gradient, {"max_it": 500, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False})
    t0 = time.perf_counter()
    _, fx = scg(x0.copy())
    el = time.perf_counter() - t0
    out["DW_single_problem"] = {"pair_ms_median": round(1e3 * float(np.median(ts)), 4), "scg_seconds": round(el, 4),
                                "scg_iterations": int(scg.stats["MaxIt"]), "fx": float(fx),
                                "through": "VarGP.free_energy + VarGP.gradient / SCG, host numpy in and out; the "
                                           "D = 1 time-parallel sweeps (small_dim.cu scan1_*)"}
    v.close()
    if with_reference:
        try:
            from baseline.refload import import_reference, reference_objects
            ref = import_reference()
            _, args = reference_objects(ref, dw)
            rv = ref["VarGP"](*args)
            rx0 = rv.initialization()
            rv.free_energy(rx0)
            rv.gradient(rx0)                         # numba kernels compiled
            rts = []
            for i in range(10):
                t0 = time.perf_counter()
                rv.free_energy(rx0)
                rv.gradient(rx0)
                rts.append(time.perf_counter() - t0)
            rscg = ref["SCG"](rv.free_energy, rv.gradient, {"max_it": 500, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False})
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                _, rfx = rscg(rx0.copy())
            out["DW_single_problem"]["reference"] = {
                "pair_ms_median": round(1e3 * float(np.median(rts)), 3), "scg_seconds": round(time.perf_counter() - t0, 3),
                "scg_iterations": int(rscg.stats["MaxIt"]), "fx": float(rfx),
                "what": "the unmodified reference (baseline/_ref, numpy/numba) on this box's CPU, same parameters"}
        except Exception as e:   # the reference is optional here (numba / scipy missing on the box)
            out["DW_single_problem"]["reference"] = {"unavailable": f"{type(e).__name__}: {e}"[:160]}

    # configs[2], the single problem: one Lorenz-63 T=2000 RK2 problem through VarGP, and its whole SCG optimisation
    sim = Simulation("bench")
    sim.setup(base("L63", "RK2", 20.0, [10.0] * 3, 2.0, 5, [10.0, 28.0, 2.6667]))
    v = sim.build()
    x0 = v.initialization()
    rng = np.random.default_rng(1)
    xs = [x0 * (1.0 + 1e-3 * rng.uniform(-1, 1, x0.size)) for _ in range(4)]
    for x_ in xs:
        v.free_energy(x_)
        v.gradient(x_)
    ts = []
    for i in range(20):
        t0 = time.perf_counter()
        v.free_energy(xs[i % 4])
        v.gradient(xs[i % 4])
        ts.append(time.perf_counter() - t0)
    scg = SCG(v.free_energy, v.gradient, {"max_it": 500, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False})
    t0 = time.perf_counter()
    _, fx = scg(x0.copy())
    el = time.perf_counter() - t0
    out["L63_single_problem"] = {"pair_ms_median": round(1e3 * float(np.median(ts)), 3), "scg_seconds": round(el, 3),
                                 "scg_iterations": int(scg.stats["MaxIt"]), "fx": float(fx),
                                 "bound": "latency (16 lanes per problem, 2 x 2001 dependent solver steps)",
                                 "through": "VarGP.free_energy + VarGP.gradient / SCG, host numpy in and out"}
    v.close()

    # configs[3]: one L96 D=40 T=1000 problem -- latency bound by 2 x T x stages dependent products
    sim = Simulation("bench")
    sim.setup(l96_params())
    v = sim.build()
    x0 = v.initialization()
    rng = np.random.default_rng(1)
    xs = [x0 * (1.0 + 1e-3 * rng.uniform(-1, 1, x0.size)) for _ in range(4)]
    for x_ in xs[:2]:
        v.free_energy(x_)
        v.gradient(x_)
    ts = []
    for i in range(12):
        t0 = time.perf_counter()
        v.free_energy(xs[i % 4])
        v.gradient(xs[i % 4])
        ts.append(time.perf_counter() - t0)
    out["L96_single_problem_latency"] = {
        "pair_ms_median": round(1e3 * float(np.median(ts)), 3), "evals_per_s": round(1.0 / float(np.median(ts)), 1),
        "bound": "latency (one CTA per sweep: 2 x 1000 steps x 2 stages of dependent 40x40x40 products)",
        "through": "VarGP.free_energy + VarGP.gradient, host numpy in and out"}
    scg = SCG(v.free_energy, v.gradient, {"max_it": 500, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False})
    n0 = v.n_eval
    t0 = time.perf_counter()
    _, fx = scg(x0.copy())
    el = time.perf_counter() - t0
    out["L96_full_scg"] = {"seconds": round(el, 3), "iterations": int(scg.stats["MaxIt"]), "fx": float(fx),
                           "cuda_evaluations": int(v.n_eval - n0),
                           "reference_seconds": "about 18 minutes on the authoring container (tests/golden/scg_L96_full.npz)"}
    v.close()
    # the same optimisation with the optimiser's vectors resident in HBM (Simulation.run(optimizer="device"))
    runs = []
    for _ in range(2):      # the first run also pays one-time costs (lazily loaded torch modules, pinned staging)
        sim2 = Simulation("bench")
        sim2.setup(l96_params())
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            sim2.run(max_it=500, display=False, optimizer="device")
        runs.append(time.perf_counter() - t0)
    out["L96_full_scg_device_optimizer"] = {"seconds": round(runs[1], 3), "first_run_seconds": round(runs[0], 3),
                                            "iterations": int(sim2.scg_stats["MaxIt"]), "fx": float(sim2.output["fx"]),
                                            "includes": "initialisation, optimisation, final evaluation with all trajectories"}
    return out


DUMP_GRAD_ROWS, DUMP_GRAD_COLS = 64, 65536


def dump_outputs(out_dir, F_all, G):
    """What the last timed step handed to its caller, for comparing two builds output for output: F of
    every problem (gathered over the ranks) as F.npy, and of this rank's gradient (54 GB at 4096
    problems) a fixed, seeded sample of 64 problems x 65536 entries (32 MB) as grad_sample.npy."""
    import torch
    rng = np.random.default_rng([SEED, 99])
    rows = np.sort(rng.choice(G.shape[0], min(DUMP_GRAD_ROWS, G.shape[0]), replace=False))
    cols = np.sort(rng.choice(G.shape[1], min(DUMP_GRAD_COLS, G.shape[1]), replace=False))
    r, c = torch.from_numpy(rows).to(G.device), torch.from_numpy(cols).to(G.device)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "F.npy", F_all.cpu().numpy())
    np.save(out / "grad_sample.npy", G[r[:, None], c[None, :]].cpu().numpy())


def run_b200(args):
    import torch
    import torch.distributed as dist
    from vgpa_b200.engine import BatchEvaluator
    from vgpa_b200.ensemble import ShardedEnsemble
    from vgpa_b200._lib import PinnedArray

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.per_gpu
    fam = l96_problem_family(rank)
    iset, arr = shard_arrays(fam, B)

    def make_evaluator(lo, hi):
        assert (lo, hi) == (rank * B, (rank + 1) * B)
        return BatchEvaluator("L96", "rk2", N_GRID, DT, [8.0], arr["sigma"], np.ones(D), fam["obs_t"], arr["obs_y"],
                              arr["m0"], fam["s0"], arr["E0"], B=B, dt_model=fam["dt_model"], device=local)
    # the sharding layer the gloo / nccl tests cover (vgpa_b200/ensemble.py): contiguous blocks of problems,
    # no data-path collective, one gather of F
    ens = ShardedEnsemble(B * world, make_evaluator, rank=rank, world=world)
    ev = ens.evaluator

    def shard_x(r, rows, fam_r, iset_r):
        """Rows [0, rows) of rank r's X = x0^{set(p)} * (1 + 0.02 u_p), u ~ U(-1, 1): generated in HBM
        (synthetic data), block by block from a per-rank seeded generator -- any rank can regenerate the
        first rows of any other rank's shard."""
        Xr = torch.empty((rows, N_X), dtype=torch.float64, device=dev)
        x0s = torch.from_numpy(np.stack([s_["x0"] for s_ in fam_r["sets"]])).to(dev)
        gen = torch.Generator(device=dev)
        gen.manual_seed(SEED % (2 ** 31) + r)
        blk = 128
        for p0 in range(0, rows, blk):
            p1 = min(rows, p0 + blk)
            u = torch.rand((blk, N_X), dtype=torch.float64, device=dev, generator=gen)[:p1 - p0] * 2.0 - 1.0
            Xr[p0:p1] = x0s[torch.from_numpy(iset_r[p0:p1]).to(dev)] * (1.0 + 0.02 * u)
            del u
        return Xr
    X = shard_x(rank, B, fam, iset)
    G = torch.empty_like(X)
    F = torch.empty(B, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    gathered = {}

    def step():
        ens.eval_device(X, F, G, stream)
        gathered["F_all"] = ens.gather_device(F)      # the only collective: gather of F (NCCL), after the status check

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    ev.sync()
    fence()
    ev.set_timing(True)
    ev.get_timing()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = ev.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    fence()
    ev.sync()
    ms = e0.elapsed_time(e1)
    clocks = sampler.summary()
    launches = ev.launch_count - launches0      # this library's kernels (the NCCL gather is not one of them)
    timing = ev.get_timing()
    ev.set_timing(False)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    F_host = F.cpu().numpy()
    assert np.all(np.isfinite(F_host)), "non-finite free energy in the bench batch"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, gathered["F_all"], G)
    value = B * world * args.steps / (ms * 1e-3)
    sharded_check = None
    if world > 1:
        # SURVEY 8(e): the sharded batch must return the single-GPU result bit for bit.  Rank 0 rebuilds the
        # first 8 problems of rank 1's shard (parameters and x), evaluates them alone and compares with what
        # the gather delivered.
        F_all = gathered["F_all"].cpu().numpy()
        assert F_all.shape == (B * world,) and np.array_equal(F_all[rank * B:(rank + 1) * B], F_host)
        if rank == 0:
            nchk = min(8, B)
            fam1 = l96_problem_family(1)
            iset1, arr1 = shard_arrays(fam1, nchk)
            X1 = shard_x(1, nchk, fam1, iset1)
            F1 = torch.empty(nchk, dtype=torch.float64, device=dev)
            with BatchEvaluator("L96", "rk2", N_GRID, DT, [8.0], arr1["sigma"], np.ones(D), fam1["obs_t"],
                                arr1["obs_y"], arr1["m0"], fam1["s0"], arr1["E0"], B=nchk,
                                dt_model=fam1["dt_model"], device=local) as ev1:
                ev1.eval_device(X1.data_ptr(), N_X, F1.data_ptr(), None, None, stream)
                ev1.sync()
            same = np.array_equal(F1.cpu().numpy(), F_all[B:B + nchk])
            sharded_check = (f"{nchk} problems of rank 1 re-evaluated on rank 0: gathered F bitwise equal" if same
                             else "MISMATCH: sharded evaluation differs from the single-GPU evaluation")
            if not same:
                print("bench.py: " + sharded_check, file=sys.stderr, flush=True)
            del X1, F1

    line = None
    if rank == 0:
        # ---- roofline of the dominant kernel (largest share of the step) -------------
        kinds = {k: v for k, v in timing.items() if k != "finalize" and v[1] > 0}
        dom = max(kinds, key=lambda k: kinds[k][0])
        tot_ms = sum(v[0] for v in timing.values())
        launches_dom = kinds[dom][1]
        avg_ms = kinds[dom][0] / launches_dom
        units_per_launch = B * N_GRID * args.steps / launches_dom   # (problem, time index) pairs
        tflops = FLOP_STEP[dom] * units_per_launch / (avg_ms * 1e-3) / 1e12
        gbs = BYTE_STEP[dom] * units_per_launch / (avg_ms * 1e-3) / 1e9
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        traffic = None
        tfiles = sorted((ROOT / "profiles").glob("traffic_r*.json"))     # newest capture that has this kernel
        tpath = next((t for t in reversed(tfiles) if dom in json.loads(t.read_text())), None)
        if tpath is not None:
            # the capture is of one 888-problem launch; `achieved` is per AVERAGE launch of the timed region
            # (4096 = 4 x 888 + 544 problems per step), so the measured bytes are scaled to the same units
            traffic = json.loads(tpath.read_text()).get(dom)
            if traffic is not None:
                traffic = float(traffic) * units_per_launch / (888.0 * N_GRID)
        roofline = {"kernel": {"fwd": "l96_fwd_kernel", "energy": "l96_energy_kernel", "bwd": "l96_bwd_kernel"}[dom],
                    "bound": "tensor", "achieved": tflops, "peak": FP64_DMMA_TFLOPS, "unit": "TFLOP/s",
                    "frac": tflops / FP64_DMMA_TFLOPS, "traffic": traffic,
                    "peak_source": "FP64 DMMA peak measured by tools/microbench.cu on this pool "
                                   "(MEASURED_PEAKS.json has no FP64 figure)",
                    "share_of_step": kinds[dom][0] / tot_ms,
                    "hbm": {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                            "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"},
                    "kernel_ms": {k: round(v[0] / max(v[1], 1), 4) for k, v in timing.items()},
                    "whole_eval": {"tflops": value / world * FLOP_EVAL / 1e12,
                                   "frac_fp64": value / world * FLOP_EVAL / 1e12 / FP64_DMMA_TFLOPS,
                                   "gbs": value / world * BYTE_EVAL / 1e9,
                                   "frac_hbm": value / world * BYTE_EVAL / 1e9 / hbm_peak}}
        line = {"metric": METRIC,
                "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": WORKLOAD,
                           "problems_per_gpu": B, "global_problems": B * world, "parallelism": f"dp{world}",
                           "l2": "inputs larger than L2 (x shard = %.1f GB)" % (B * N_X * 8 / 1e9),
                           "chunk": ev.chunk_size},
                "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline}
        if sharded_check:
            line["sharded_equals_single_gpu"] = sharded_check

    # ---- e2e: the same evaluation through the public host API with HOST buffers ----
    # 1024 problems per step (27 GB of pinned host memory per rank) when the box has the memory for
    # every rank, else 512: the pipeline's fill / drain (first H2D, last kernels + D2H, ~27 ms) is a
    # fixed cost per call, so the longer step measures the steady state of the API more closely
    Be = args.e2e_problems
    if Be <= 0:
        avail_gb = 0.0
        try:
            with open("/proc/meminfo") as fh:
                for ln in fh:
                    if ln.startswith("MemAvailable:"):
                        avail_gb = float(ln.split()[1]) / 1e6
        except OSError:
            pass
        Be = 1024 if avail_gb >= 64.0 * world else 512
        if world > 1:   # every rank must use the same step size: take the smallest choice
            tb = torch.tensor([Be], dtype=torch.int64, device=dev)
            dist.all_reduce(tb, op=dist.ReduceOp.MIN)
            Be = int(tb.item())
    Be = min(Be, B)
    xe = PinnedArray((Be, N_X))
    ge = PinnedArray((Be, N_X))
    xe.array[:] = X[:Be].cpu().numpy()
    ev.close()
    del X, G
    torch.cuda.empty_cache()
    ev_e = BatchEvaluator("L96", "rk2", N_GRID, DT, [8.0], arr["sigma"][:Be], np.ones(D), fam["obs_t"],
                          arr["obs_y"][:Be], arr["m0"][:Be], fam["s0"], arr["E0"][:Be], B=Be,
                          dt_model=fam["dt_model"], device=local,
                          # 64-problem chunks: H2D of chunk c+1, kernels of chunk c and D2H of chunk c-1 overlap
                          scratch_bytes=64 * 8 * N_GRID * (2 * D + 2 * D * D + 1) + 1024)
    Fe = np.empty(Be)
    for _ in range(2):
        ev_e.eval(xe.array, True, Fe, ge.array)
    fence()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        ev_e.eval(xe.array, True, Fe, ge.array)
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    te = torch.tensor([el], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = Be * world * args.e2e_steps / float(te.item())
    assert np.allclose(Fe, F_host[:Be], rtol=1e-12, atol=0.0), "host-API result differs from device-API result"
    ev_e.close()
    xe.free()
    ge.free()

    ceiling = copy_ceiling(torch, dist, dev, world)
    scg_line = None
    if args.scg_problems > 0:
        scg_line = ensemble_scg(torch, dist, dev, local, rank, world, fam, args.scg_problems)
    if rank == 0:
        e2e_gbs = e2e_val * N_X * 8.0 / 1e9           # per direction: x in, gradient out
        line["e2e"] = {"value": e2e_val, "unit": "evals/s", "h2d_bytes_per_step": int(Be * N_X * 8),
                       "d2h_bytes_per_step": int(Be * N_X * 8 + Be * 8),
                       "sample": f"{Be} problems per GPU per step through vgpa_eval with pinned host x/grad, "
                                 f"{args.e2e_steps} steps",
                       "gbs_per_direction": e2e_gbs, "copy_ceiling_gbs": ceiling,
                       "frac_of_copy_ceiling": e2e_gbs / ceiling,
                       "copy_ceiling_how": "1 GiB pinned H2D + 1 GiB pinned D2H cudaMemcpyAsync concurrently on two "
                                           "streams, all ranks at once, GB/s per direction summed over ranks"}
        if world == 1:
            threads = len(os.sched_getaffinity(0))
            probs = max(threads, 1) * (12 if threads <= 16 else (6 if threads <= 64 else 3))   # ~10-30 s of CPU work
            rate, el_cpu = cpu_port_rate(threads, probs, fam)
            line["cpu_baseline"] = {"value": rate, "unit": "evals/s", "cores": threads, "kind": "port",
                                    "sample": f"{probs} L96 N=1001 problems, one OpenMP thread each, "
                                              f"{el_cpu:.1f} s of wall time (oracle/vgpa_oracle.c)"}
            if not args.no_python_reference:
                # the unmodified reference on this box's CPU, on ensemble member (set 0, sigma = 4.0, x = x0),
                # and the CUDA path on the SAME problem at the SAME x: a live parity check
                s0_ = fam["sets"][0]
                cal = reference_python_rate({"obs_y": s0_["obs_y"], "m0": s0_["m0"]})
                if "unavailable" not in cal:
                    xr, gr = cal.pop("x0"), cal.pop("grad")
                    with BatchEvaluator("L96", "rk2", N_GRID, DT, [8.0], np.full(D, 4.0), np.ones(D), fam["obs_t"],
                                        s0_["obs_y"], s0_["m0"], fam["s0"], s0_["E0"], B=1, dt_model=fam["dt_model"],
                                        device=local) as ev1:
                        Fg, Gg = ev1.eval(xr)
                    na = N_GRID * D * D
                    cal["cuda_vs_reference"] = {
                        "F_rel": abs(float(Fg[0]) - cal["F_x0"]) / abs(cal["F_x0"]),
                        "dL_dA_rel": float(np.abs(Gg[0][:na] - gr[:na]).max() / np.abs(gr[:na]).max()),
                        "dL_db_rel": float(np.abs(Gg[0][na:] - gr[na:]).max() / np.abs(gr[na:]).max()),
                        "x0_equal": bool(np.array_equal(xr, s0_["x0"]))}
                line["cpu_baseline_reference"] = cal
            if not args.no_secondary:
                try:
                    line["secondary"] = secondary_configs(torch, local, hbm_peak, with_reference=not args.no_python_reference)
                except Exception as e:      # never lose the headline line to a secondary measurement
                    line["secondary"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        if scg_line is not None:
            line["ensemble_scg"] = scg_line
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--per-gpu", type=int, default=PER_GPU, help="problems per GPU (default 4096)")
    ap.add_argument("--e2e-problems", type=int, default=0, help="problems per e2e step (0 = 1024 if host memory allows, else 512)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-python-reference", action="store_true",
                    help="skip the one warm evaluation of the unmodified Python reference (about a minute of CPU)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the other BASELINE configs (N = 1 only)")
    ap.add_argument("--scg-problems", type=int, default=444,
                    help="problems per GPU of the device-resident ensemble OPTIMISATION (secondary key ensemble_scg; 0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write F and a seeded sample of the gradient of the last timed step to DIR/*.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
