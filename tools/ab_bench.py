"""A/B comparison of two or more builds of the project in one session on one GPU.

    python tools/ab_bench.py --out DIR [--rounds 3] [--dump] TREE_A TREE_B [...] -- <bench.py arguments>

Every TREE is a copy of the repository with librbm_b200.so already built in it (`python -m rigid_body_manipulation_b200.build`);
a parent commit is exported with `git archive <rev> | tar -x -C ab_trees/<name>` (ab_trees/ is git-ignored).  The trees run
`python bench.py <arguments>` in turn, A B ... A B ..., for --rounds rounds, so that clock and neighbour drift hit every tree alike.
With --dump each run also writes its outputs (bench.py --dump-outputs) and the last round's outputs of every tree are compared with
the first tree's.

Written under DIR: lines.jsonl (every bench line, tagged with tree and round), summary.json (the card's name, power limit and maximum
SM clock, read once with a read-only nvidia-smi query; median / min / max of value, extra.rnea_f32.value and e2e.value per tree; the
output comparison), and the summary again on stdout.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

FIELDS = {"value": ("value",), "rnea_f32": ("extra", "rnea_f32", "value"), "e2e": ("e2e", "value")}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True,
                             timeout=60).stdout
        return out.strip().splitlines()
    except (OSError, subprocess.TimeoutExpired) as e:
        return [f"nvidia-smi unavailable: {e}"]


def dig(line, path):
    for k in path:
        if not isinstance(line, dict) or k not in line:
            return None
        line = line[k]
    return line


def compare_dumps(ref_dir, dir_):
    """name -> max |delta| / max |ref| over the whole array, and whether the two arrays are bit-identical"""
    out = {}
    for name in sorted(os.listdir(ref_dir)):
        a, b = np.load(os.path.join(ref_dir, name)), np.load(os.path.join(dir_, name))
        if a.shape != b.shape:
            out[name] = {"shape_mismatch": [list(a.shape), list(b.shape)]}
            continue
        scale = float(np.abs(a).max()) or 1.0
        out[name] = {"max_abs_delta_over_max_abs": float(np.abs(a.astype(np.float64) - b).max() / scale), "bit_identical": bool(np.array_equal(a, b))}
    return out


def main():
    argv = sys.argv[1:]
    bench_args = []
    if "--" in argv:
        i = argv.index("--")
        argv, bench_args = argv[:i], argv[i + 1:]
    ap = argparse.ArgumentParser()
    ap.add_argument("trees", nargs="+")
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--dump", action="store_true", help="pass --dump-outputs to bench.py and compare the outputs of the trees")
    ap.add_argument("--timeout", type=float, default=1800.0, help="seconds per bench.py run")
    args = ap.parse_args(argv)
    if len(args.trees) < 2:
        ap.error("give at least two trees")
    trees = [os.path.abspath(t) for t in args.trees]
    for t in trees:
        if not os.path.exists(os.path.join(t, "rigid_body_manipulation_b200", "librbm_b200.so")):
            ap.error(f"{t}: librbm_b200.so is not built")
    labels = [os.path.basename(t.rstrip("/")) for t in trees]
    if len(set(labels)) != len(labels):
        ap.error("the trees' directory names must differ")
    out = os.path.abspath(args.out)
    os.makedirs(out, exist_ok=True)
    summary = {"card": card(), "bench_args": bench_args, "rounds": args.rounds, "trees": dict(zip(labels, trees))}
    lines = {lb: [] for lb in labels}
    with open(os.path.join(out, "lines.jsonl"), "a") as log:
        for r in range(args.rounds):
            for tree, lb in zip(trees, labels):
                extra = ["--dump-outputs", os.path.join(out, "dumps", lb, f"r{r}")] if args.dump else []
                p = subprocess.run([sys.executable, "bench.py", *bench_args, *extra], cwd=tree, capture_output=True, text=True, timeout=args.timeout)
                got = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
                rec = {"tree": lb, "round": r, "returncode": p.returncode}
                if p.returncode != 0 or not got:
                    rec["stderr_tail"] = p.stderr[-2000:]
                else:
                    rec["line"] = json.loads(got[-1])
                    lines[lb].append(rec["line"])
                log.write(json.dumps(rec) + "\n")
                log.flush()
                print(f"round {r} {lb}: rc {p.returncode} value {dig(rec.get('line'), ('value',))}", flush=True)
    stats = {}
    for lb in labels:
        stats[lb] = {"runs": len(lines[lb])}
        for key, path in FIELDS.items():
            v = [x for x in (dig(ln, path) for ln in lines[lb]) if x is not None]
            if v:
                stats[lb][key] = {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v)), "n": len(v)}
    base = labels[0]
    for lb in labels[1:]:
        for key in FIELDS:
            if key in stats[lb] and key in stats[base]:
                stats[lb][key]["median_over_" + base] = stats[lb][key]["median"] / stats[base][key]["median"]
    summary["stats"] = stats
    if args.dump:
        last = f"r{args.rounds - 1}"
        ref = os.path.join(out, "dumps", base, last)
        summary["outputs_vs_" + base] = {lb: compare_dumps(ref, os.path.join(out, "dumps", lb, last)) for lb in labels[1:]
                                         if os.path.isdir(ref) and os.path.isdir(os.path.join(out, "dumps", lb, last))}
    with open(os.path.join(out, "summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
