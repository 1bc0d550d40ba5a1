#!/usr/bin/env python
"""A/B of bench.py between a base commit and the working tree, on one GPU, in one session.

  python tools/ab_bench.py export [--rev HEAD] [--dir ab_base]
      exports the base commit with `git archive` into DIR (ignored by git) and builds its library there, so the GPU
      machine only has to run it.
  python tools/ab_bench.py run [--base ab_base] [--runs 3] [--steps 20] [--warmup 3] [--out ab_out]
      runs `bench.py --gpus 1` from the two trees alternately (base, new, base, new, ...), each run a separate process
      that exits; the first run of each tree also writes --dump-outputs, and the two dumps are compared element for
      element.  K1 alone (tools/bench_repack.py) runs once per tree.  Records the card's name, power limit and max SM
      clock (nvidia-smi, query only) and prints one JSON object: per tree the median / min / max of ms_per_step, value,
      value_from_resident_u8.ms_per_step, e2e.ms_per_step and every config's ms, whether every new run was faster than
      every base run, and the dump comparison.  Raw bench lines go to OUT/runs.jsonl."""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def export(args):
    d = os.path.abspath(os.path.join(ROOT, args.dir))
    if os.path.exists(d):
        raise SystemExit(f"{d} exists: remove it first")
    os.makedirs(d)
    arc = subprocess.run(["git", "-C", ROOT, "archive", args.rev], check=True, capture_output=True).stdout
    subprocess.run(["tar", "-x", "-C", d], input=arc, check=True)
    subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=d, check=True)
    print(json.dumps({"exported": args.rev, "dir": d}))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def bench_once(tree, args, dump=None):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.steps), "--warmup", str(args.warmup),
           "--skip-cpu"] + args.bench_args
    if dump:
        cmd += ["--dump-outputs", dump]
    p = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    if p.returncode != 0 or not lines:
        return {"error": f"rc={p.returncode}", "stderr_tail": p.stderr[-2000:]}
    return json.loads(lines[-1])


def metrics(line):
    out = {}
    if "error" in line:
        return out
    out["ms_per_step"] = line.get("ms_per_step")
    out["value"] = line.get("value")
    out["value_from_resident_u8.ms_per_step"] = (line.get("value_from_resident_u8") or {}).get("ms_per_step")
    out["e2e.ms_per_step"] = (line.get("e2e") or {}).get("ms_per_step")
    out["roofline.ms_per_launch"] = (line.get("roofline") or {}).get("ms_per_launch")
    out["roofline.padded_bytes_per_launch"] = (line.get("roofline") or {}).get("padded_bytes_per_launch")
    for c in line.get("configs") or []:
        if c.get("ms") is not None:
            out[c["config"] + ".ms"] = c["ms"]
    strong = line.get("strong") or {}
    if strong.get("ms_per_step") is not None:
        out["strong.ms_per_step"] = strong["ms_per_step"]
    return out


def stats(runs):
    keys = sorted({k for r in runs for k in r})
    out = {}
    for k in keys:
        v = [r[k] for r in runs if r.get(k) is not None]
        if v:
            out[k] = {"median": statistics.median(v), "min": min(v), "max": max(v), "n": len(v)}
    return out


def compare_dumps(a, b):
    fa = sorted(f for f in os.listdir(a) if f.endswith(".npy")) if os.path.isdir(a) else []
    fb = sorted(f for f in os.listdir(b) if f.endswith(".npy")) if os.path.isdir(b) else []
    if not fa or fa != fb:
        return {"identical": False, "files_base": fa, "files_new": fb}
    diff = {}
    for f in fa:
        x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
        if x.shape != y.shape or not np.array_equal(x, y):
            diff[f] = int(np.sum(x != y)) if x.shape == y.shape else "shape"
    return {"identical": not diff, "files": fa, "differing": diff}


def run(args):
    out = os.path.abspath(args.out)
    os.makedirs(out, exist_ok=True)
    trees = {"base": os.path.abspath(os.path.join(ROOT, args.base)), "new": ROOT}
    info = gpu_info()
    raw = open(os.path.join(out, "runs.jsonl"), "w")
    per = {"base": [], "new": []}
    dumps = tempfile.mkdtemp(prefix="ab_dumps_")  # full-size dumps: compared here, not kept
    for i in range(args.runs):
        for name, tree in trees.items():
            dump = os.path.join(dumps, name) if i == 0 else None
            line = bench_once(tree, args, dump)
            raw.write(json.dumps({"tree": name, "run": i, "line": line}) + "\n")
            raw.flush()
            per[name].append(metrics(line))
    repack = {}
    for name, tree in trees.items():
        p = subprocess.run([sys.executable, "tools/bench_repack.py"], cwd=tree, capture_output=True, text=True)
        lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
        repack[name] = json.loads(lines[-1]) if lines else {"error": p.stderr[-2000:]}
    base_ms = [r["ms_per_step"] for r in per["base"] if r.get("ms_per_step")]
    new_ms = [r["ms_per_step"] for r in per["new"] if r.get("ms_per_step")]
    summary = {
        "gpu": info, "runs_per_tree": args.runs, "steps": args.steps, "warmup": args.warmup,
        "base": stats(per["base"]), "new": stats(per["new"]),
        "new_over_base_median_ms_per_step": (statistics.median(new_ms) / statistics.median(base_ms))
        if base_ms and new_ms else None,
        "every_new_run_faster": bool(base_ms and new_ms and max(new_ms) < min(base_ms)),
        "bench_repack": repack,
        "dumps": compare_dumps(os.path.join(dumps, "base"), os.path.join(dumps, "new")),
    }
    shutil.rmtree(dumps, ignore_errors=True)
    with open(os.path.join(out, "ab.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps(summary))


def main():
    ap = argparse.ArgumentParser()
    sub = ap.add_subparsers(dest="cmd", required=True)
    e = sub.add_parser("export")
    e.add_argument("--rev", default="HEAD")
    e.add_argument("--dir", default="ab_base")
    r = sub.add_parser("run")
    r.add_argument("--base", default="ab_base")
    r.add_argument("--runs", type=int, default=3)
    r.add_argument("--steps", type=int, default=20)
    r.add_argument("--warmup", type=int, default=3)
    r.add_argument("--out", default="ab_out")
    r.add_argument("bench_args", nargs="*", help="extra bench.py arguments (after --)")
    args = ap.parse_args()
    export(args) if args.cmd == "export" else run(args)


if __name__ == "__main__":
    main()
