"""Cost of final observations and device-side partial resets (sf_list_finished, sf_reset_finished,
sf_observe_list) on one GPU; prints one JSON line.

Workload: the squad5v5 configuration of bench.py (Squad, levels 1-10, default capacities, episodes truncated at
2,048 steps, the 28-symbol synthetic action stream), 131,072 arenas.  Two handles on the same seeds, one with
auto_reset = 1 ("auto") and one with auto_reset = 0 ("manual"), go through bench.py's untimed set-up (--setup
steps; the arenas spread over episode ages by 16 staggered partial resets, applied to both).  Then, for --steps
steps, timed with CUDA events around each call (pass 1):
  list_finished         sf_list_finished alone, on the manual handle after its step (before the reset)
  observe_list_finished sf_observe_list of the arenas that finished in that step (ids and device count from
                        sf_list_finished, n_max = --n-max), player observation, [32][31][31]
  observe_all           sf_observe of every arena, the same observation (every --observe-every steps)
and for --steps more steps, the order of the two handles alternating (pass 2):
  step_auto             sf_step of the auto handle
  step_manual_reset     sf_step + sf_reset_finished of the manual handle (the same trajectory, checked at the end)
After the loop, on the state it left (no more stepping), --reps alternating repetitions of:
  observe_list k random ids for k in --ks, and all ids in order, both layouts, next to observe_all in both
  reset_today           the path a caller has without these calls for the finished arenas of one step: the status
                        column of sf_step_out to the host, the ids picked there, sf_reset with the host ids
                        (it synchronises); host clock around it.  Compared with sf_reset_finished on the same
                        finished set: sf_save of the terminal arenas before, sf_load between the two.
Observation rates are bytes of observations written per second (123,008 B per observation).
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

OBS_BYTES = sfcfg.OBS_LEN * 4


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    return e0, e1


def summary(ms):
    return dict(ms=round(statistics.median(ms), 4), ms_mean=round(statistics.fmean(ms), 4), ms_min=round(min(ms), 4),
                ms_max=round(max(ms), 4), n=len(ms))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--setup", type=int, default=2048, help="untimed set-up steps (age spreading, as bench.py --prewarm)")
    ap.add_argument("--steps", type=int, default=256, help="timed steps")
    ap.add_argument("--n-max", type=int, default=16384, help="rows of the finished-arena observation buffer")
    ap.add_argument("--observe-every", type=int, default=8)
    ap.add_argument("--ks", default="1024,13107,131072")
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_final_obs.py measures the GPU kernels; no CUDA device is usable")
    n = args.envs
    n_max = min(args.n_max, n)
    kw = dict(mode="Squad", level=1, level_max=10, squad_agents=False, max_steps=2048)
    auto, manual = BatchedArena(n, auto_reset=True, **kw), BatchedArena(n, auto_reset=False, **kw)
    dev = auto.device
    table = sfcfg.ACTIONS28
    # ---- untimed set-up, as bench.py: 16 buckets of arenas reset at staggered steps
    t, buckets = 0, 16
    per = max(1, args.setup // buckets)
    ids_all = np.arange(n, dtype=np.int32)
    for j in range(buckets):
        for _ in range(per):
            act = auto.synth_actions(t, table)
            auto.step(act)
            manual.step(act)
            manual.reset_finished()
            t += 1
        if j + 1 < buckets:
            for sim in (auto, manual):
                sim.reset(ids_all[ids_all % buckets == j])
    torch.cuda.synchronize()
    assert torch.equal(auto.state_hash(), manual.state_hash()), "the two handles parted during the set-up"
    # ---- timed steps
    ids = torch.empty(n, dtype=torch.int32, device=dev)
    count = torch.empty(1, dtype=torch.int32, device=dev)
    fin_obs = torch.empty((n_max, 1, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN), device=dev)
    all_obs = torch.empty((n, 1, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN), device=dev)
    acts = torch.empty((n, auto.n_agents), dtype=torch.uint8, device=dev)
    ev = {k: [] for k in ("step_auto", "step_manual_reset", "list_finished", "observe_list_finished", "observe_all")}
    finished = []
    for s in range(args.steps):
        acts.copy_(auto.synth_actions(t, table))
        t += 1
        auto.step(acts)  # pass 1 times the calls between the step and the reset; pass 2 the step and the reset
        manual.step(acts)
        ev["list_finished"].append(event_ms(lambda: manual.list_finished(ids, count)))
        ev["observe_list_finished"].append(event_ms(lambda: manual.observe(1, out=fin_obs, env_ids=ids[:n_max], count=count)))
        finished.append(count.clone())
        if s % args.observe_every == 0:
            ev["observe_all"].append(event_ms(lambda: manual.observe(1, out=all_obs)))
        manual.reset_finished()
    for s in range(args.steps):  # pass 2, the order of the two handles alternating
        acts.copy_(auto.synth_actions(t, table))
        t += 1
        if s % 2:
            ev["step_auto"].append(event_ms(lambda: auto.step(acts)))
            ev["step_manual_reset"].append(event_ms(lambda: (manual.step(acts), manual.reset_finished())))
        else:
            ev["step_manual_reset"].append(event_ms(lambda: (manual.step(acts), manual.reset_finished())))
            ev["step_auto"].append(event_ms(lambda: auto.step(acts)))
    torch.cuda.synchronize()
    ms = {k: [a.elapsed_time(b) for a, b in v] for k, v in ev.items()}
    fin = torch.cat(finished).cpu().numpy()
    assert torch.equal(auto.state_hash(), manual.state_hash()), "auto-reset and sf_reset_finished parted"
    assert torch.equal(auto.step_out(), manual.step_out())
    assert auto.stats() == manual.stats()
    res = {k: summary(v) for k, v in ms.items()}
    over = res["step_manual_reset"]["ms"] - res["step_auto"]["ms"]
    res["reset_overhead"] = dict(ms=round(over, 4), pct=round(100 * over / res["step_auto"]["ms"], 2),
                                 mean_ms=round(res["step_manual_reset"]["ms_mean"] - res["step_auto"]["ms_mean"], 4))
    res["finished_per_step"] = dict(mean=round(float(fin.mean()), 1), median=float(np.median(fin)), max=int(fin.max()),
                                    beyond_n_max=int((fin > n_max).sum()))
    res["observe_list_finished"]["vs_observe_all"] = round(res["observe_list_finished"]["ms"] / res["observe_all"]["ms"], 4)
    # ---- observe_list of k ids on the state as it stands
    rng = np.random.default_rng(3)
    ks = [int(k) for k in args.ks.split(",")]
    lists = {"random_%d" % k: torch.as_tensor(rng.integers(0, n, min(k, n)).astype(np.int32), device=dev) for k in ks}
    lists["all_in_order"] = torch.arange(n, dtype=torch.int32, device=dev)
    flat = all_obs.view(-1)
    obs_cases = {}
    for cl in (False, True):
        tag = "nhwc" if cl else "nchw"
        obs_cases["observe_all_" + tag] = (lambda cl=cl: manual.observe(1, out=all_obs, channels_last=cl), n)
        for name, li in lists.items():
            k = li.numel()
            out = flat[:k * sfcfg.OBS_LEN].view(k, 1, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN)
            obs_cases["observe_list_%s_%s" % (name, tag)] = (
                lambda cl=cl, li=li, out=out: manual.observe(1, out=out, channels_last=cl, env_ids=li), k)
    for fn, _ in obs_cases.values():
        fn()
    oms = {k: [] for k in obs_cases}
    for _ in range(args.reps):
        evs = {k: event_ms(fn) for k, (fn, _) in obs_cases.items()}
        torch.cuda.synchronize()
        for k, (a, b) in evs.items():
            oms[k].append(a.elapsed_time(b))
    obs_res = {}
    for k, (_, rows) in obs_cases.items():
        r = summary(oms[k])
        r["rows"] = rows
        r["bytes_per_s"] = round(rows * OBS_BYTES / (r["ms"] * 1e-3) / 1e9, 1) * 1e9
        obs_res[k] = r
    for k, r in obs_res.items():
        tag = k.rsplit("_", 1)[1]
        full = obs_res["observe_all_" + tag]["ms"]
        r["vs_observe_all"] = round(r["ms"] / full, 4)
        r["rows_share"] = round(r["rows"] / n, 4)
    res["observe"] = obs_res
    # ---- the reset path a caller has today, on the same finished sets as sf_reset_finished
    today, device_reset, sets = [], [], []
    for _ in range(args.reps * 4):
        acts.copy_(auto.synth_actions(t, table))
        t += 1
        manual.step(acts)
        host_ids = np.nonzero(manual.step_out()[:, 0].cpu().numpy() != sfcfg.RUNNING)[0].astype(np.int32)
        if host_ids.size == 0:
            manual.reset_finished()
            continue
        rec = manual.save(host_ids)
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        ids_h = np.nonzero(manual.step_out()[:, 0].cpu().numpy() != sfcfg.RUNNING)[0].astype(np.int32)
        manual.reset(ids_h)
        today.append((time.perf_counter() - h0) * 1e3)
        manual.load(rec, host_ids)
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        manual.reset_finished()
        torch.cuda.synchronize()
        device_reset.append((time.perf_counter() - h0) * 1e3)
        sets.append(int(host_ids.size))
    if today:
        res["reset_today"] = dict(summary(today), finished=int(np.median(sets)), clock="host, synchronised")
        res["reset_finished_same_sets"] = dict(summary(device_reset), clock="host, synchronised")
    print(json.dumps(dict(metric="final observations and device-side partial resets", envs=n, setup_steps=args.setup,
                          timed_steps=args.steps, n_max=n_max, cases=res, device=torch.cuda.get_device_name(),
                          power_limit_w=power_limit_w(),
                          goals=dict(reset_overhead_within_3pct=bool(res["reset_overhead"]["pct"] <= 3.0),
                                     observe_list_all_within_3pct=bool(
                                         obs_res["observe_list_all_in_order_nchw"]["vs_observe_all"] <= 1.03 and
                                         obs_res["observe_list_all_in_order_nhwc"]["vs_observe_all"] <= 1.03)))))
    auto.close(), manual.close()


if __name__ == "__main__":
    main()
