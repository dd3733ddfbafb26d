"""Cost of the device-list record calls (sf_save_list / sf_load_list) against sf_save / sf_load on one GPU, and what
they take out of a search loop; writes one JSON file (--out, default profiles/r06_record_list.json) and prints it.

Workload: the squad5v5 configuration of bench.py (Squad, levels 1-10, default capacities, episodes truncated at
2,048 steps, auto-reset), 131,072 arenas after --setup steps of the 28-symbol synthetic action stream.

Kernel cases, each one call timed with CUDA events around it, the order rotating from one repetition to the next
(--reps after --warmup; medians).  Every load writes back the records the same arenas were saved into, so the state
does not move during the measurement:
  save_all / load_all                 sf_save / sf_load of all arenas (env_ids NULL)
  save_list_all / load_list_all       sf_save_list / sf_load_list of every id in order (count = NULL)
  save_list_K / load_list_K           a random list of K distinct ids, K in --ks (K = n_envs: a permutation)
  save_K / load_K                     the same lists through sf_save / sf_load with host ids (staging included)
Wall-clock cases (host clock around the call and a device synchronise, medians of --reps):
  broadcast_device    one root into --slots slots: sf_save_list of the root, sf_load_list with rows = zeros
  broadcast_host      BatchedArena.clone([root] * slots, slots): sf_save + sf_load with host ids (synchronising)
  expansion_graph     one search expansion replayed from a CUDA graph: device broadcast of the root into the slots,
                      4 x (sf_observe_list of the player + sf_step_list of the slots), restore of the slots from the
                      root record (sf_load_list, rows = zeros)
  expansion_eager     the same expansion with host-id clone and host-id restore (sf_save / sf_load), the
                      observe_list / step_list calls as above
Each path is checked once against its reference at this size (records byte for byte, the expansion's hashes).
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_snapshot import power_limit_w  # noqa: E402
from strikeforce_b200 import config as sfcfg  # noqa: E402
from strikeforce_b200.sim import BatchedArena  # noqa: E402

KW = dict(mode="Squad", level=1, level_max=10, squad_agents=False, max_steps=2048, auto_reset=True)
EXPANSION_STEPS = 4


def _stats(v):
    return dict(ms=round(statistics.median(v), 4), ms_min=round(min(v), 4), ms_max=round(max(v), 4), n=len(v))


def kernel_cases(cases, reps, warmup):
    names = list(cases)
    ms = {c: [] for c in names}
    for r in range(warmup + reps):
        order = names[r % len(names):] + names[:r % len(names)]
        for c in order:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            cases[c]()
            e1.record()
            e1.synchronize()
            if r >= warmup:
                ms[c].append(e0.elapsed_time(e1))
    return {c: _stats(v) for c, v in ms.items()}


def wall_cases(cases, reps, warmup):
    names = list(cases)
    ms = {c: [] for c in names}
    for r in range(warmup + reps):
        order = names[r % len(names):] + names[:r % len(names)]
        for c in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            cases[c]()
            torch.cuda.synchronize()
            if r >= warmup:
                ms[c].append(1e3 * (time.perf_counter() - t0))
    return {c: _stats(v) for c, v in ms.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--setup", type=int, default=1024, help="steps before the measurement")
    ap.add_argument("--ks", default="131072,4096,32")
    ap.add_argument("--slots", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_record_list.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_record_list.py measures the GPU kernels; no CUDA device is usable")
    n, table = args.envs, sfcfg.ACTIONS28
    sim = BatchedArena(n, **KW)
    dev, B = sim.device, sim.snapshot_bytes
    for t in range(args.setup):
        sim.step(sim.synth_actions(t, table))
    t = args.setup
    rng = np.random.default_rng(7)
    every = torch.arange(n, dtype=torch.int32, device=dev)
    rec = sim.save()
    buf = torch.empty_like(rec)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    # ---- checks at this size
    assert torch.equal(sim.save(every, out=buf), rec), "save_list of all ids differs from sf_save"
    assert int(sim.load(buf, every, status=status)) == 0 and torch.equal(sim.save(), rec), "load_list of all ids"
    cases = {"save_all": lambda: sim.save(out=rec),
             "save_list_all": lambda: sim.save(every, out=buf),
             "load_all": lambda: sim.load(rec),
             "load_list_all": lambda: sim.load(buf, every, status=status)}
    ks = [min(int(k), n) for k in args.ks.split(",")]
    for k in ks:
        ids_h = rng.choice(n, k, replace=False).astype(np.int32)
        ids = torch.as_tensor(ids_h, device=dev)
        out = torch.empty((k, B), dtype=torch.uint8, device=dev)  # a buffer per list: its loads put back what it saved
        assert torch.equal(sim.save(ids, out=out), rec[ids.long()]), "save_list of %d random ids" % k
        cases["save_list_%d" % k] = lambda ids=ids, out=out: sim.save(ids, out=out)
        cases["load_list_%d" % k] = lambda ids=ids, out=out: sim.load(out, ids, status=status)
        cases["save_%d" % k] = lambda ids_h=ids_h, out=out: sim.save(ids_h, out=out)
        cases["load_%d" % k] = lambda ids_h=ids_h, out=out: sim.load(out, ids_h)
    res = kernel_cases(cases, args.reps, args.warmup)
    assert int(status) == 0 and torch.equal(sim.save(), rec), "a timed load moved the state"
    for c in ("save_list_all", "load_list_all"):
        res[c]["vs_" + c.replace("_list", "")] = round(res[c]["ms"] / res[c.replace("_list", "")]["ms"], 4)
    for c in ("save_list_all", "save_all", "load_list_all", "load_all"):
        res[c]["record_tb_per_s"] = round(n * B / res[c]["ms"] / 1e9, 3)
    for k in ks:
        for kind in ("save", "load"):
            res["%s_list_%d" % (kind, k)]["vs_host_ids"] = round(res["%s_list_%d" % (kind, k)]["ms"] / res["%s_%d" % (kind, k)]["ms"], 4)
    # ---- one root into the slots, and one search expansion
    K, root = args.slots, 0
    slots_h = (1 + rng.choice(n - 1, K, replace=False)).astype(np.int32)
    slots = torch.as_tensor(slots_h, device=dev)
    root_id = torch.tensor([root], dtype=torch.int32, device=dev)
    zeros = torch.zeros(K, dtype=torch.int32, device=dev)
    root_rec = torch.empty((1, B), dtype=torch.uint8, device=dev)
    act = sim.synth_actions(t, table)[:K].contiguous()
    obs = torch.empty((K, 1, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN), device=dev)

    def broadcast_device():
        sim.save(root_id, out=root_rec)
        sim.load(root_rec, slots, rows=zeros, status=status)

    def broadcast_host():
        sim.clone([root] * K, slots_h)

    def expand(clone, restore):
        clone()
        for _ in range(EXPANSION_STEPS):
            sim.observe(1, out=obs, env_ids=slots)
            sim.step_list(act, slots)
        restore()

    def expansion_device():
        expand(broadcast_device, lambda: sim.load(root_rec, slots, rows=zeros, status=status))

    host_rows = np.zeros(K, np.int32)

    def expansion_eager():
        expand(broadcast_host, lambda: sim.load(root_rec, slots_h, rows=host_rows))

    # the device expansion against the host one: same hashes after one of each from the same state
    sim.load(rec)
    expansion_device()
    h_dev = sim.state_hash().clone()
    assert int(status) == 0
    sim.load(rec)
    expansion_eager()
    assert torch.equal(sim.state_hash(), h_dev), "device-list expansion parted from the host-id one"
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    launches = sim.launches
    with torch.cuda.graph(graph, stream=stream):
        expansion_device()
    captured = sim.launches - launches
    torch.cuda.current_stream().wait_stream(stream)
    sim.load(rec)
    graph.replay()
    assert torch.equal(sim.state_hash(), h_dev), "graph replay of the expansion"
    wall = wall_cases({"broadcast_device": broadcast_device, "broadcast_host": broadcast_host,
                       "expansion_graph": graph.replay, "expansion_eager": expansion_eager}, args.reps, args.warmup)
    wall["broadcast_device"]["vs_host"] = round(wall["broadcast_device"]["ms"] / wall["broadcast_host"]["ms"], 4)
    wall["expansion_graph"]["vs_eager"] = round(wall["expansion_graph"]["ms"] / wall["expansion_eager"]["ms"], 4)
    wall["expansion_graph"]["captured_launches"] = captured
    out = dict(metric="sf_save_list / sf_load_list against sf_save / sf_load", envs=n, setup_steps=args.setup,
               record_bytes=B, reps=args.reps, device=torch.cuda.get_device_name(), power_limit_w=power_limit_w(),
               kernel_cases=res, wall_cases=wall, slots=K, expansion_steps=EXPANSION_STEPS,
               goals=dict(save_list_all_within_3pct=bool(res["save_list_all"]["vs_save_all"] <= 1.03),
                          load_list_all_within_3pct=bool(res["load_list_all"]["vs_load_all"] <= 1.03)))
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    sim.close()


if __name__ == "__main__":
    main()
