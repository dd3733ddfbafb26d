#!/usr/bin/env python
"""A/B of two builds of the library on the step-kernel benchmark, alternated in one process tree so that both see
the same card, clocks and neighbours.

    python tools/ab_step.py A.so B.so [--rounds 5] [--out DIR] [-- bench.py arguments]

Every round runs `bench.py --steps 50 --warmup 5 --no-cpu --no-obs` (or the arguments after `--`) once with A and
once with B (SF_LIB_PATH), alternating which goes first, and reads `ms_per_step` from its JSON line.  The card's
name, power limit and SM clock are read with nvidia-smi before every run; the SM clock bench.py sampled during
its timed steps is kept with every run.  With --out, every run also writes
--dump-outputs into DIR/<A|B><round>, and the tool checks that all of them are identical: the same steps of the
same workload give the same results whatever the build.  Prints one JSON line: per build the runs, median, min,
max and spread (max - min), and B's median against A's."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMI_Q = "name,power.limit,clocks.sm,clocks.max.sm"


def smi():
    r = subprocess.run(["nvidia-smi", "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0],
                        "--query-gpu=" + SMI_Q, "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
    return dict(zip(SMI_Q.split(","), [x.strip() for x in r.stdout.strip().split(",")])) if r.returncode == 0 else {}


def run(lib, bench_args, dump):
    env = dict(os.environ, SF_LIB_PATH=os.path.abspath(lib))
    cmd = [sys.executable, os.path.join(ROOT, "bench.py")] + bench_args + (["--dump-outputs", dump] if dump else [])
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=1800)
    if r.returncode != 0:
        sys.exit("bench.py failed with %s:\n%s" % (lib, r.stderr[-4000:]))
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line["ms_per_step"], line.get("clocks")


def load_dump(d):
    return {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def main():
    argv = sys.argv[1:]
    bench_args = ["--steps", "50", "--warmup", "5", "--no-cpu", "--no-obs"]
    if "--" in argv:
        i = argv.index("--")
        argv, bench_args = argv[:i], argv[i + 1:]
    ap = argparse.ArgumentParser()
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", help="write and compare --dump-outputs of every run under this directory")
    args = ap.parse_args(argv)
    libs = {"A": args.a, "B": args.b}
    ms = {"A": [], "B": []}
    clocks = {"A": [], "B": []}
    cards = []
    dumps = []
    for r in range(args.rounds):
        for name in ("AB" if r % 2 == 0 else "BA"):
            cards.append(smi())
            dump = os.path.join(args.out, "%s%d" % (name, r)) if args.out else None
            t, c = run(libs[name], bench_args, dump)
            ms[name].append(t)
            clocks[name].append(c)
            if dump:
                dumps.append(dump)
            print("round %d %s %.4f ms/step  %s" % (r, name, ms[name][-1], cards[-1]), file=sys.stderr, flush=True)
    same = None
    if dumps:
        first = load_dump(dumps[0])
        same = all(sorted(x) == sorted(first) and all(np.array_equal(x[k], first[k]) for k in first)
                   for x in map(load_dump, dumps[1:]))
    res = {"bench_args": bench_args, "gpu": cards[0].get("name"), "power_limit": cards[0].get("power.limit"),
           "clocks_sm": sorted({c.get("clocks.sm") for c in cards}), "clocks_max_sm": cards[0].get("clocks.max.sm")}
    for name in "AB":
        v = ms[name]
        res[name] = {"lib": libs[name], "ms_per_step": v, "median": statistics.median(v), "min": min(v), "max": max(v),
                     "spread": max(v) - min(v), "timed_clocks": clocks[name]}
    res["B_over_A"] = res["B"]["median"] / res["A"]["median"]
    if same is not None:
        res["outputs_identical"] = same
    print(json.dumps(res))
    if same is False:
        sys.exit("the builds' outputs differ")


if __name__ == "__main__":
    main()
