"""Throughput of arena records (sf_save / sf_load) on one GPU; prints one JSON line.

Workload: the squad5v5 configuration of bench.py (Squad, levels 1-10, default capacities, episodes truncated at
2,048 steps, auto-reset), 131,072 arenas after --setup steps of the 28-symbol synthetic action stream, so that
the state is not young.  Cases, each timed with CUDA events around every call after a warm-up (the calls
synchronise; the time covers the staging of the id lists and every kernel of the call):
  save_all      sf_save of all arenas in order
  load_all      sf_load of all arenas in order
  save_perm / load_perm   the same for a random permutation of all ids (reported only)
  clone_4096    one root into 4,096 slots: sf_save of the root, sf_load with rows (BatchedArena.clone)
For comparison, a torch device-to-device copy of the same byte count as the all-arenas record buffer is timed
in the same process.  Rates are record bytes per second (each byte is read once and written once).
"""
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


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return statistics.median(ms), min(ms), max(ms)


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
        return float(out.strip().splitlines()[0])
    except Exception:  # no nvidia-smi on the host: the number is reported as unknown
        return None


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--setup", type=int, default=1024, help="steps before the measurement")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--clone-slots", type=int, default=4096)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_snapshot.py measures the GPU kernels; no CUDA device is usable")
    n = args.envs
    sim = BatchedArena(n, mode="Squad", level=1, level_max=10, squad_agents=False, auto_reset=True, max_steps=2048)
    for t in range(args.setup):
        sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
    torch.cuda.synchronize()
    B = sim.snapshot_bytes
    rec = torch.empty((n, B), dtype=torch.uint8, device=sim.device)
    stats0 = sim.stats()
    hash0 = sim.state_hash()
    perm = np.random.default_rng(1).permutation(n).astype(np.int32)
    slots = min(args.clone_slots, n - 1)
    root, dst = 0, np.arange(1, slots + 1, dtype=np.int32)
    cases = {
        "save_all": (lambda: sim.save(out=rec), n),
        "load_all": (lambda: sim.load(rec), n),
        "save_perm": (lambda: sim.save(perm, out=rec), n),
        "load_perm": (lambda: sim.load(rec, perm), n),
    }
    res = {}
    for name, (fn, count) in cases.items():
        if name == "load_all":
            sim.save(out=rec)  # the records of the arenas as they stand: every load is a no-op on the state
        med, lo, hi = timed(fn, args.reps, args.warmup)
        res[name] = dict(ms=round(med, 4), ms_min=round(lo, 4), ms_max=round(hi, 4), records=count,
                         bytes_per_s=count * B / (med * 1e-3))
    assert torch.equal(sim.state_hash(), hash0), "loading the arenas' own records changed them"
    med, lo, hi = timed(lambda: sim.clone(np.full(slots, root, np.int32), dst), args.reps, args.warmup)
    res["clone_%d" % slots] = dict(ms=round(med, 4), ms_min=round(lo, 4), ms_max=round(hi, 4), records=slots,
                                   bytes_per_s=(slots + 1) * B / (med * 1e-3))
    assert sim.stats() == stats0, "save / load changed the statistics"
    del rec
    src = torch.empty(n * B, dtype=torch.uint8, device=sim.device)
    dst_buf = torch.empty_like(src)
    src.fill_(1)
    med, lo, hi = timed(lambda: dst_buf.copy_(src), args.reps, args.warmup)
    copy = dict(ms=round(med, 4), ms_min=round(lo, 4), ms_max=round(hi, 4), bytes=n * B, bytes_per_s=n * B / (med * 1e-3))
    for r in res.values():
        r["vs_copy"] = round(r["bytes_per_s"] / copy["bytes_per_s"], 3)
        r["bytes_per_s"] = round(r["bytes_per_s"] / 1e9, 1) * 1e9
    copy["bytes_per_s"] = round(copy["bytes_per_s"] / 1e9, 1) * 1e9
    print(json.dumps(dict(metric="arena records per second", envs=n, setup_steps=args.setup, record_bytes=B,
                          cases=res, torch_d2d_copy=copy, device=torch.cuda.get_device_name(),
                          power_limit_w=power_limit_w(), target_met=bool(min(res["save_all"]["vs_copy"],
                                                                              res["load_all"]["vs_copy"]) >= 2 / 3))))
    sim.close()


if __name__ == "__main__":
    main()
