"""Cost of sf_action_mask on one GPU, beside one step and one observation of the same arenas; writes one JSON file
(--out, default profiles/r07_action_mask.json) and prints it.

Workload: the squad5v5 configuration of bench.py (Squad, levels 1-10, default capacities, episodes truncated at
2,048 steps, auto-reset), 131,072 arenas after --setup steps of the 28-symbol synthetic action stream.

Cases, each one call timed with CUDA events around it, the order rotating from one repetition to the next (--reps
after --warmup; medians):
  mask_all        sf_action_mask of every arena (env_ids NULL)
  mask_list_K     sf_action_mask of a random list of K distinct ids, K in --ks
  step            one sf_step of all arenas (the state moves on: the masks are of a state one step apart each time)
  observe         one fp32 channels-last sf_observe of the player of all arenas
The card name, its power limit and its SM clock are read in the same run.  The mask of all arenas is checked once
against the list form at this size."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from strikeforce_b200 import config as sfcfg  # noqa: E402
from strikeforce_b200.sim import BatchedArena  # noqa: E402

KW = dict(mode="Squad", level=1, level_max=10, squad_agents=False, max_steps=2048, auto_reset=True)


def smi(field):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=" + field,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
        return float(out.strip().splitlines()[0])
    except Exception:  # no nvidia-smi on the host: the number is reported as unknown
        return None


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--setup", type=int, default=1024, help="steps before the measurement")
    ap.add_argument("--ks", default="4096,32")
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_action_mask.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_action_mask.py measures the GPU kernels; no CUDA device is usable")
    n, table = args.envs, sfcfg.ACTIONS28
    sim = BatchedArena(n, **KW)
    dev = sim.device
    for t in range(args.setup):
        sim.step(sim.synth_actions(t, table))
    t = args.setup
    rng = np.random.default_rng(7)
    mask = torch.empty((n, sim.n_agents), dtype=torch.int32, device=dev)
    obs = torch.empty((n, 1, sfcfg.OBS_WIN, sfcfg.OBS_WIN, sfcfg.OBS_CH), device=dev)
    act = sim.synth_actions(t, table).clone()
    every = torch.arange(n, dtype=torch.int32, device=dev)
    assert torch.equal(sim.action_mask(every), sim.action_mask(out=mask)), "mask of all ids differs from the list form"
    words = mask.cpu().numpy().view(np.uint32)
    cases = {"mask_all": lambda: sim.action_mask(out=mask),
             "step": lambda: sim.step(act),
             "observe": lambda: sim.observe(1, out=obs, channels_last=True)}
    for k in [min(int(k), n) for k in args.ks.split(",")]:
        ids = torch.as_tensor(rng.choice(n, k, replace=False).astype(np.int32), device=dev)
        out = torch.empty((k, sim.n_agents), dtype=torch.int32, device=dev)
        cases["mask_list_%d" % k] = lambda ids=ids, out=out: sim.action_mask(ids, out=out)
    names = list(cases)
    ms = {c: [] for c in names}
    for r in range(args.warmup + args.reps):
        for c in names[r % len(names):] + names[:r % len(names)]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            cases[c]()
            e1.record()
            e1.synchronize()
            if r >= args.warmup:
                ms[c].append(e0.elapsed_time(e1))
    res = {c: dict(ms=round(statistics.median(v), 4), ms_min=round(min(v), 4), ms_max=round(max(v), 4), n=len(v))
           for c, v in ms.items()}
    res["mask_all"]["vs_step"] = round(res["mask_all"]["ms"] / res["step"]["ms"], 4)
    res["mask_all"]["vs_observe"] = round(res["mask_all"]["ms"] / res["observe"]["ms"], 4)
    live = words[words != 0]
    out = dict(metric="sf_action_mask against sf_step and sf_observe of the same arenas", envs=n, setup_steps=args.setup,
               reps=args.reps, device=torch.cuda.get_device_name(), power_limit_w=smi("power.limit"),
               sm_clock_mhz=smi("clocks.sm"), cases=res,
               mean_bits_per_controllable_slot=round(float(np.mean([bin(int(w)).count("1") for w in live])), 3),
               goals=dict(mask_all_below_10pct_of_step=bool(res["mask_all"]["vs_step"] <= 0.10)))
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    sim.close()


if __name__ == "__main__":
    main()
