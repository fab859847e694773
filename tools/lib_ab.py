"""
A/B of two builds of libvgpa_b200.so on the flagship workload of bench.py.

    python tools/lib_ab.py OLD.so NEW.so [--runs 3] [--steps 10] [--warmup 3] [--out DIR]

Runs `bench.py --no-python-reference --no-secondary --scg-problems 0 --dump-outputs ...` with VGPA_LIB pointing
at each library in turn, alternating the arms (old new, new old, old new, ...) so that a drift of the machine
does not favour one of them.  Prints the card's name and power limit, each run's `value` and per-kernel CUDA-event
times (`roofline.kernel_ms`), per arm the median and spread, and whether F.npy and grad_sample.npy are
byte-identical between the arms and between the runs of one arm.  The summary also goes to
DIR/lib_ab.json.

Build the old library from the parent commit in a separate checkout (`python -m vgpa_b200.build` there) and pass
the path of its libvgpa_b200.so.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def run_bench(lib, dump, args):
    cmd = [sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", str(args.steps), "--warmup",
           str(args.warmup), "--no-python-reference", "--no-secondary", "--scg-problems", "0", "--dump-outputs", str(dump)]
    env = dict(os.environ, VGPA_LIB=str(Path(lib).resolve()))
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout[-4000:] + r.stderr[-4000:])
        raise SystemExit(f"bench.py failed with {lib}")
    line = next(ln for ln in reversed(r.stdout.splitlines()) if ln.startswith("{"))
    return json.loads(line)


def same_files(a, b):
    return all((a / f).read_bytes() == (b / f).read_bytes() for f in ("F.npy", "grad_sample.npy"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="where the dumps and lib_ab.json go (default: a new temporary directory)")
    args = ap.parse_args()
    out = Path(args.out) if args.out else Path(tempfile.mkdtemp(prefix="lib_ab_"))
    out.mkdir(parents=True, exist_ok=True)
    info = gpu_info()
    print(f"gpu: {info}", flush=True)
    libs = {"old": args.old, "new": args.new}
    runs = {"old": [], "new": []}
    for r in range(args.runs):
        for arm in (("old", "new") if r % 2 == 0 else ("new", "old")):
            res = run_bench(libs[arm], out / f"{arm}{r}", args)
            km = res["roofline"]["kernel_ms"]
            runs[arm].append({"value": res["value"], "kernel_ms": km, "clocks": res.get("clocks")})
            print(f"run {r} {arm}: value {res['value']:.1f} evals/s, kernel_ms {json.dumps(km)}", flush=True)
    summary = {"gpu": info, "steps": args.steps, "warmup": args.warmup, "runs": runs}
    for arm, rs in runs.items():
        v = [x["value"] for x in rs]
        s = {"value_median": statistics.median(v), "value_min": min(v), "value_max": max(v),
             "value_spread_pct": 100.0 * (max(v) - min(v)) / statistics.median(v)}
        for k in rs[0]["kernel_ms"]:
            s[f"{k}_ms_median"] = statistics.median(x["kernel_ms"][k] for x in rs)
        summary[arm] = s
        print(f"{arm}: {json.dumps(s)}", flush=True)
    summary["value_gain_pct"] = 100.0 * (summary["new"]["value_median"] / summary["old"]["value_median"] - 1.0)
    summary["outputs_identical_old_vs_new"] = same_files(out / "old0", out / "new0")
    summary["outputs_identical_within_arms"] = all(same_files(out / f"{a}0", out / f"{a}{r}")
                                                   for a in runs for r in range(1, args.runs))
    print(f"value gain {summary['value_gain_pct']:+.2f} %; F.npy and grad_sample.npy identical old vs new: "
          f"{summary['outputs_identical_old_vs_new']}, within arms: {summary['outputs_identical_within_arms']}", flush=True)
    (out / "lib_ab.json").write_text(json.dumps(summary, indent=1))
    if not summary["outputs_identical_old_vs_new"]:
        raise SystemExit("the two libraries compute different outputs")


if __name__ == "__main__":
    main()
