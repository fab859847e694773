"""
Cost of per-problem observation schedules: F + gradient evaluations of a shared-schedule handle (vgpa_create) against a
ragged handle (vgpa_create_obs_rows) with the same total number of observations, and against the workaround the
ragged handle replaces (one handle per distinct schedule).

    python tools/obs_rows_bench.py [--reps 5] [--only l96,l96d64,l63,ou1k,ou64k,workaround]

The shared handle observes every `every`-th grid index.  The ragged handle's counts are drawn around the same mean
(uniform in [M/2, 3M/2], then adjusted so that the totals agree) and its indices are random sorted subsets of the
grid, seeded.  Both handles evaluate the same x rows with the same scratch budget (the same pass split).  Each
timing is the median of --reps calls, alternated between the variants, after one warm-up call of each; CUDA events
bracket each call on one stream.  Prints one JSON line with the card's name and power limit.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


# name: model, method, D, N, B, observe every, problems per pass (0: the default budget)
WORKLOADS = {
    "l96": ("L96", "rk2", 40, 1001, 4096, 10, 888),
    "l96d64": ("L96", "rk2", 64, 1001, 512, 10, 256),
    "l63": ("L63", "rk2", 3, 2002, 4096, 20, 0),
    "ou1k": ("OU", "rk4", 1, 1001, 1024, 20, 0),
    "ou64k": ("OU", "rk4", 1, 1001, 65536, 20, 0),
}
THETA = {"DW": [1.0], "OU": [2.0], "L63": [10.0, 28.0, 8.0 / 3.0], "L96": [8.0]}


def ragged_schedules(N, B, M, rng):
    """B sorted index sets inside (0, N - 1) with counts around M and B * M indices in all."""
    lo, hi = max(1, M // 2), min(N - 2, (3 * M) // 2)
    counts = rng.integers(lo, hi + 1, B)
    diff = B * M - int(counts.sum())
    while diff != 0:
        p = int(rng.integers(B))
        step = 1 if diff > 0 else -1
        if lo <= counts[p] + step <= hi:
            counts[p] += step
            diff -= step
    return [np.sort(rng.choice(np.arange(1, N - 1), size=int(c), replace=False)) for c in counts]


def make(model, method, D, N, B, obs_t, rng, idx=None, scratch=0):
    """A handle over problems idx (all when None): obs_t one shared index array, or a list of B arrays."""
    from vgpa_b200.engine import BatchEvaluator
    idx = np.arange(B) if idx is None else np.asarray(idx)
    if isinstance(obs_t, list):
        obs_t = [obs_t[p] for p in idx]
        obs_y = [np.sin(0.01 * t[:, None] + np.arange(D)) for t in obs_t]
    else:
        obs_y = np.broadcast_to(np.sin(0.01 * obs_t[:, None] + np.arange(D)), (len(idx), obs_t.size, D)).copy()
    return BatchEvaluator(model, method, N, 0.01, THETA[model], np.full(D, 0.5 if D > 1 else 0.8), np.full(D, 0.5),
                          obs_t, obs_y, np.zeros(D), (0.2 * np.eye(D)).ravel(), 0.0, B=len(idx), dt_model=0.01, D=D,
                          scratch_bytes=scratch)


def timed(torch, fns, reps):
    """Median milliseconds of each fn: one warm-up call each, then `reps` rounds calling them in turn."""
    for f in fns:
        f()
    torch.cuda.synchronize()
    ts = [[] for _ in fns]
    for _ in range(reps):
        for k, f in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            b.synchronize()
            ts[k].append(a.elapsed_time(b))
    return [float(np.median(t)) for t in ts]


def x_rows(torch, ev, B):
    """x for B problems: the initialization of the first handle, perturbed per problem (seeded)."""
    n = ev.n_x
    X = torch.empty((B, n), dtype=torch.float64, device="cuda")
    ev.initialization_device(X.data_ptr(), n, 0.0)
    torch.cuda.synchronize()
    g = torch.Generator(device="cuda").manual_seed(0)
    for lo in range(0, B, 64):     # in slices: a (B, n) temporary would not fit next to x at L96 x 4096
        Xs = X[lo:lo + 64]
        Xs.mul_(1.0 + 0.01 * torch.randn(Xs.shape, generator=g, device="cuda", dtype=torch.float64))
    return X


def evaluate(ev, X, F, G, lo=0):
    n = ev.n_x
    ev.eval_device(X[lo].data_ptr(), n, F[lo].data_ptr(), G[lo].data_ptr(), n)


def run_pair(torch, name, reps):
    model, method, D, N, B, every, per_pass = WORKLOADS[name]
    rng = np.random.default_rng([1, B, N])
    shared_t = np.arange(every // 2, N - 1, every, dtype=np.int64)
    M = shared_t.size
    rag_t = ragged_schedules(N, B, M, rng)
    scratch = per_pass * 8 * N * (2 * D + 2 * D * D + 1) + 64 if per_pass else 0
    with make(model, method, D, N, B, shared_t, rng, scratch=scratch) as e_s, \
            make(model, method, D, N, B, rag_t, rng, scratch=scratch) as e_r:
        assert e_s.chunk_size == e_r.chunk_size
        X = x_rows(torch, e_s, B)
        F = torch.empty(B, dtype=torch.float64, device="cuda")
        G = torch.empty_like(X)
        t_s, t_r = timed(torch, [lambda: evaluate(e_s, X, F, G), lambda: evaluate(e_r, X, F, G)], reps)
        e_s.sync()
        e_r.sync()
        ok = bool(torch.isfinite(F).all().item())
        chunk = e_s.chunk_size
        del X, G, F
        torch.cuda.empty_cache()
    return {"workload": name, "model": model, "method": method, "D": D, "N": N, "B": B, "problems_per_pass": chunk,
            "obs_per_problem_mean": M, "ragged_counts_min_max": [int(min(t.size for t in rag_t)),
                                                                 int(max(t.size for t in rag_t))],
            "shared_ms": round(t_s, 3), "ragged_ms": round(t_r, 3), "ragged_over_shared": round(t_r / t_s, 4),
            "finite": ok}


def run_workaround(torch, B, n_sched, reps):
    """L96 D = 40, RK2, N = 1001: one ragged handle against one handle per distinct schedule (problems grouped by
    schedule, so each handle's rows are a contiguous slice of x)."""
    D, N, every = 40, 1001, 10
    rng = np.random.default_rng([2, B, n_sched])
    M = np.arange(every // 2, N - 1, every).size
    distinct = ragged_schedules(N, n_sched, M, rng)
    per = B // n_sched
    rag_t = [distinct[p // per] for p in range(B)]
    handles = [make("L96", "rk2", D, N, B, rag_t, rng, idx=np.arange(k * per, (k + 1) * per)) for k in range(n_sched)]
    with make("L96", "rk2", D, N, B, rag_t, rng) as e_r:
        X = x_rows(torch, e_r, B)
        F = torch.empty(B, dtype=torch.float64, device="cuda")
        G = torch.empty_like(X)

        def per_schedule():
            for k, ev in enumerate(handles):
                evaluate(ev, X, F, G, k * per)

        t_r, t_w = timed(torch, [lambda: evaluate(e_r, X, F, G), per_schedule], reps)
        e_r.sync()
        for ev in handles:
            ev.sync()
        del X, G, F
    for ev in handles:
        ev.close()
    torch.cuda.empty_cache()
    return {"workload": f"workaround-{n_sched}-schedules", "model": "L96", "method": "rk2", "D": D, "N": N, "B": B,
            "handles": n_sched, "ragged_ms": round(t_r, 3), "one_handle_per_schedule_ms": round(t_w, 3),
            "ragged_evals_per_s": round(1e3 * B / t_r, 1), "per_schedule_evals_per_s": round(1e3 * B / t_w, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="l96,l96d64,l63,ou1k,ou64k,workaround")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("obs_rows_bench: no CUDA device")
    out = {"card": card(), "runs": []}
    for name in a.only.split(","):
        if name == "workaround":
            rs = [run_workaround(torch, 1024, 8, a.reps), run_workaround(torch, 256, 256, a.reps)]
        else:
            rs = [run_pair(torch, name, a.reps)]
        for r in rs:
            out["runs"].append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
