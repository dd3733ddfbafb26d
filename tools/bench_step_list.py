"""Cost of sf_step_list (stepping a device list of arenas) against sf_step on one GPU; writes one JSON file
(--out, default profiles/r05_step_list.json) and prints it.

Workload: the squad5v5 configuration of bench.py (Squad, levels 1-10, default capacities, episodes truncated at
2,048 steps, the 28-symbol synthetic action stream), 131,072 arenas, after bench.py's untimed set-up (--setup steps;
the arenas spread over episode ages by 16 staggered partial resets).  A twin handle takes the same set-up; after it,
one sf_step of the twin is checked against sf_step_list of all ids in order and then of a random permutation on the
measured handle (state hashes, sf_step_out, statistics).

Cases, each one call timed with CUDA events, the order of the cases rotating from one repetition to the next
(--reps repetitions after --warmup untimed ones; medians reported; every call advances the arenas it steps):
  step                    sf_step of all arenas
  list_all_in_order       sf_step_list of every id in order (count = NULL)
  list_all_permuted       sf_step_list of a random permutation of every id
  list_K_contiguous       sf_step_list of K consecutive ids, for K in --ks
  list_K_random           sf_step_list of K distinct random ids
  handle_K                sf_step of a separate handle of K arenas loaded (sf_load) with the K contiguous arenas'
                          state: what a caller does without sf_step_list, without the save / load it also needs
Small K is bounded by the serial chain of one warp (DESIGN.md section 2), not by K / n_envs.
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_snapshot import power_limit_w  # noqa: E402
from strikeforce_b200 import config as sfcfg  # noqa: E402
from strikeforce_b200.sim import BatchedArena  # noqa: E402

KW = dict(mode="Squad", level=1, level_max=10, squad_agents=False, max_steps=2048)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--setup", type=int, default=2048, help="untimed set-up steps (age spreading, as bench.py --prewarm)")
    ap.add_argument("--ks", default="13107,4096,1024,32")
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_step_list.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_step_list.py measures the GPU kernels; no CUDA device is usable")
    n = args.envs
    sim, twin = BatchedArena(n, auto_reset=True, **KW), BatchedArena(n, auto_reset=True, **KW)
    dev, table = sim.device, sfcfg.ACTIONS28
    # ---- untimed set-up, as bench.py: 16 buckets of arenas reset at staggered steps
    t, buckets = 0, 16
    per = max(1, args.setup // buckets)
    ids_all = np.arange(n, dtype=np.int32)
    for j in range(buckets):
        for _ in range(per):
            act = sim.synth_actions(t, table)
            sim.step(act)
            twin.step(act)
            t += 1
        if j + 1 < buckets:
            for s in (sim, twin):
                s.reset(ids_all[ids_all % buckets == j])
    every = torch.arange(n, dtype=torch.int32, device=dev)
    rng = np.random.default_rng(7)
    perm = torch.as_tensor(rng.permutation(n).astype(np.int32), device=dev)
    # ---- the same trajectory through sf_step and sf_step_list at this size
    for ids in (every, perm):
        act = sim.synth_actions(t, table)
        twin.step(act)
        sim.step_list(act[ids.long()].contiguous(), ids)
        t += 1
        assert torch.equal(sim.state_hash(), twin.state_hash()), "sf_step_list parted from sf_step"
        assert torch.equal(sim.step_out(), twin.step_out())
    assert sim.stats() == twin.stats()
    twin.close()
    # ---- the cases
    ks = [int(k) for k in args.ks.split(",")]
    acts = torch.empty((n, sim.n_agents), dtype=torch.uint8, device=dev)
    cases = {"step": lambda: sim.step(acts),
             "list_all_in_order": lambda: sim.step_list(acts, every),
             "list_all_permuted": lambda: sim.step_list(acts, perm)}
    handles = {}
    for k in ks:
        start = (n - k) // 2 // 32 * 32
        contiguous = every[start:start + k].contiguous()
        random = torch.as_tensor(np.sort(rng.choice(n, k, replace=False)).astype(np.int32), device=dev)
        rows = acts[:k]
        cases["list_%d_contiguous" % k] = lambda rows=rows, ids=contiguous: sim.step_list(rows, ids)
        cases["list_%d_random" % k] = lambda rows=rows, ids=random: sim.step_list(rows, ids)
        h = BatchedArena(k, auto_reset=True, **KW)
        h.load(sim.save(np.arange(start, start + k)))
        handles[k] = h
        cases["handle_%d" % k] = lambda h=h, rows=rows: h.step(rows)
    names = list(cases)
    ms = {c: [] for c in names}
    launches = {}
    for r in range(args.warmup + args.reps):
        acts.copy_(sim.synth_actions(t, table))
        t += 1
        order = names[r % len(names):] + names[:r % len(names)]
        ev = {}
        for c in order:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = sim.launches
            e0.record()
            cases[c]()
            e1.record()
            ev[c] = (e0, e1)
            launches[c] = sim.launches - l0
        torch.cuda.synchronize()
        if r >= args.warmup:
            for c, (e0, e1) in ev.items():
                ms[c].append(e0.elapsed_time(e1))
    res = {}
    for c in names:
        v = ms[c]
        res[c] = dict(ms=round(statistics.median(v), 4), ms_min=round(min(v), 4), ms_max=round(max(v), 4), n=len(v),
                      launches=launches[c] if not c.startswith("handle_") else 1)
    step = res["step"]["ms"]
    for c in ("list_all_in_order", "list_all_permuted"):
        res[c]["vs_step"] = round(res[c]["ms"] / step, 4)
    for k in ks:
        for kind in ("contiguous", "random"):
            c = "list_%d_%s" % (k, kind)
            res[c]["vs_handle_%d" % k] = round(res[c]["ms"] / res["handle_%d" % k]["ms"], 4)
            res[c]["vs_step"] = round(res[c]["ms"] / step, 4)
    out = dict(metric="sf_step_list against sf_step", envs=n, setup_steps=args.setup, reps=args.reps,
               device=torch.cuda.get_device_name(), power_limit_w=power_limit_w(), cases=res,
               goals=dict(all_in_order_within_3pct=bool(res["list_all_in_order"]["vs_step"] <= 1.03),
                          contiguous_within_10pct_of_a_k_handle={
                              str(k): bool(res["list_%d_contiguous" % k]["vs_handle_%d" % k] <= 1.10) for k in ks}))
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    for h in handles.values():
        h.close()
    sim.close()


if __name__ == "__main__":
    main()
