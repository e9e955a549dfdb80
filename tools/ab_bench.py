"""A/B benchmark of two source trees: time the headline and check that both compute the same thing.

  git archive <base-rev> | tar -x -C .ab_base && python .ab_base/__graft_entry__.py   # once, on the build machine
  python tools/ab_bench.py [--base .ab_base] [--new .] [--rounds 3] [--steps 20] [--out DIR]

Each tree runs its OWN bench.py (which resolves the library from its own location) as
`bench.py --no-secondary --no-cpu-baseline --steps K`, alternating base and new (A B A B ...), so that drift in clocks
or in other work on the host hits both alike.  Then each tree runs once more with `--dump-outputs`, and every .npy
file of the two dumps is compared with np.array_equal.  Prints the card name and power limit, every JSON line, the
median ratio new/base, and a summary line; writes the dumps and ab.json under --out (default: a new temporary
directory); exits non-zero when the outputs differ.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(tree, steps, extra=()):
    cmd = [sys.executable, os.path.join(os.path.abspath(tree), "bench.py"), "--gpus", "1", "--no-secondary",
           "--no-cpu-baseline", "--steps", str(steps)] + list(extra)
    out = subprocess.run(cmd, capture_output=True, text=True)
    if out.returncode != 0:
        sys.stderr.write(out.stderr)
        raise SystemExit("ab_bench: %s failed with exit code %d" % (" ".join(cmd), out.returncode))
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    return json.loads(lines[-1])


def compare_dumps(a, b):
    import numpy as np
    names = sorted(set(os.listdir(a)) | set(os.listdir(b)))
    diff = []
    for n in names:
        pa, pb = os.path.join(a, n), os.path.join(b, n)
        if not (os.path.exists(pa) and os.path.exists(pb)) or not np.array_equal(np.load(pa), np.load(pb)):
            diff.append(n)
    return names, diff


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", default=os.path.join(ROOT, ".ab_base"))
    ap.add_argument("--new", default=ROOT)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", help="directory for the dumps and ab.json (default: a new temporary directory)")
    args = ap.parse_args()
    args.out = args.out or tempfile.mkdtemp(prefix="ab_bench_")
    os.makedirs(args.out, exist_ok=True)
    print("output: " + args.out)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    print("gpu: " + " | ".join(l.strip() for l in smi.stdout.strip().splitlines()))

    runs = {"base": [], "new": []}
    for r in range(args.rounds):
        for tag, tree in (("base", args.base), ("new", args.new)):
            line = run_bench(tree, args.steps)
            runs[tag].append(line)
            print("%s round %d: %s" % (tag, r, json.dumps(line)), flush=True)

    dumps = {}
    for tag, tree in (("base", args.base), ("new", args.new)):
        dumps[tag] = os.path.join(os.path.abspath(args.out), "dump_" + tag)
        run_bench(tree, 1, ["--dump-outputs", dumps[tag]])
    names, diff = compare_dumps(dumps["base"], dumps["new"])
    counts = __import__("numpy").load(os.path.join(dumps["new"], "counts.npy"))

    vb = [l["value"] for l in runs["base"]]
    vn = [l["value"] for l in runs["new"]]
    summary = {
        "base_values": vb, "new_values": vn,
        "base_ms_per_step": [l["ms_per_step"] for l in runs["base"]],
        "new_ms_per_step": [l["ms_per_step"] for l in runs["new"]],
        "median_ratio": statistics.median(vn) / statistics.median(vb),
        "every_new_faster_than_every_base": min(vn) > max(vb),
        "outputs_compared": len(names), "outputs_differing": diff,
        "new_counts_last_step": [float(x) for x in counts],
    }
    print("summary: " + json.dumps(summary))
    json.dump({"runs": runs, "summary": summary, "gpu": smi.stdout}, open(os.path.join(args.out, "ab.json"), "w"), indent=1)
    return 1 if diff else 0


if __name__ == "__main__":
    sys.exit(main())
