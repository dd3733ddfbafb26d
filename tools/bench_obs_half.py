"""Half-precision observations written by the observation kernel (SF_OBS_F16 / SF_OBS_BF16) against fp32, and
against today's path to a half tensor (fp32 sf_observe, then .to(dtype)), on one GPU; prints one JSON line.

Workload: the squad5v5 configuration of bench.py (Squad, levels 1-10, default capacities, episodes truncated at
2,048 steps, the 28-symbol synthetic action stream), 131,072 arenas, the player's observation, after the untimed
set-up of tools/bench_final_obs.py (--setup steps; the arenas spread over episode ages by 16 staggered resets).
On the state that leaves, --reps repetitions (at least 7) alternate over every case, each timed with CUDA events:
  observe_<layout>_<format>_<path>  layout nchw ([32][31][31]) or nhwc (SF_OBS_NHWC); format fp32, fp16 or bf16;
                                     path all (sf_observe of every arena) or list (sf_observe_list of --list random
                                     ids)
  cast_<layout>_<format>_all         fp32 sf_observe of every arena, then .to(dtype)
  forward_<format>_<input>           for scale only, reduced precision: one AgentModel forward of --fwd-batch
                                     observations under torch.autocast(dtype), channels-last, fed the half NHWC
                                     observations (input half) or the fp32 NHWC observations (input fp32)
Medians are reported; rates are observation bytes written per second (123,008 B fp32, 61,504 B half).  The
observation buffers (16 GB fp32 at the default size) are far larger than L2.  Before the timing, every half output
is compared with the cast fp32 output of the same state, bit for bit; a mismatch fails the script.
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
from strikeforce_b200 import policy  # noqa: E402
from strikeforce_b200.sim import BatchedArena  # noqa: E402

FORMATS = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--setup", type=int, default=2048, help="untimed set-up steps (age spreading, as bench.py --prewarm)")
    ap.add_argument("--list", type=int, default=13107, help="random ids of the sf_observe_list path")
    ap.add_argument("--fwd-batch", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_obs_half.py measures the GPU kernels; no CUDA device is usable")
    assert args.reps >= 7
    n = args.envs
    sim = BatchedArena(n, mode="Squad", level=1, level_max=10, squad_agents=False, auto_reset=True, max_steps=2048)
    dev = sim.device
    # ---- untimed set-up, as tools/bench_final_obs.py: 16 buckets of arenas reset at staggered steps
    t, buckets = 0, 16
    per = max(1, args.setup // buckets)
    ids_all = np.arange(n, dtype=np.int32)
    for j in range(buckets):
        for _ in range(per):
            sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
            t += 1
        if j + 1 < buckets:
            sim.reset(ids_all[ids_all % buckets == j])
    torch.cuda.synchronize()
    rng = np.random.default_rng(5)
    lst = torch.as_tensor(rng.integers(0, n, args.list).astype(np.int32), device=dev)
    rows = {"all": n, "list": args.list}
    shape = {"nchw": lambda r: (r, 1, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN),
             "nhwc": lambda r: (r, 1, sfcfg.OBS_WIN, sfcfg.OBS_WIN, sfcfg.OBS_CH)}
    bufs = {f: torch.empty(n * sfcfg.OBS_LEN, dtype=dt, device=dev) for f, dt in FORMATS.items()}

    def obs(layout, fmt, path):
        r = rows[path]
        out = bufs[fmt][:r * sfcfg.OBS_LEN].view(shape[layout](r))
        return sim.observe(1, out=out, channels_last=layout == "nhwc", dtype=FORMATS[fmt],
                           env_ids=lst if path == "list" else None)

    # ---- the half outputs equal the cast fp32 outputs at the timed size
    checked = 0
    for layout in shape:
        for path in rows:
            for fmt in ("fp16", "bf16"):
                ref = obs(layout, "fp32", path).to(FORMATS[fmt])
                got = obs(layout, fmt, path)
                if not torch.equal(got.view(torch.int16), ref.view(torch.int16)):
                    sys.exit("MISMATCH: %s %s %s differs from the cast fp32 observation" % (layout, fmt, path))
                checked += ref.numel()
                del ref
    torch.cuda.synchronize()
    # ---- the cases
    cases = {}
    for layout in shape:
        for fmt in FORMATS:
            for path in rows:
                cases["observe_%s_%s_%s" % (layout, fmt, path)] = (lambda a=layout, b=fmt, c=path: obs(a, b, c),
                                                                   rows[path] * sfcfg.OBS_LEN * FORMATS[fmt].itemsize)
        for fmt in ("fp16", "bf16"):
            cases["cast_%s_%s_all" % (layout, fmt)] = (lambda a=layout, b=fmt: obs(a, "fp32", "all").to(FORMATS[b]),
                                                       n * sfcfg.OBS_LEN * 2)
    B = min(args.fwd_batch, n)
    model = policy.AgentModel().to(dev).eval().to(memory_format=torch.channels_last)
    state = model.initial_state(B, dev)
    # the forward's inputs: copies of the first B observations (channels-last), so a forward times the model alone
    xs = {f: obs("nhwc", f, "all")[:B].flatten(0, 1).clone() for f in FORMATS}
    for fmt in ("fp16", "bf16"):
        for inp in (fmt, "fp32"):
            def fwd(fmt=fmt, x=xs[inp]):
                with torch.no_grad(), torch.autocast("cuda", dtype=FORMATS[fmt]):
                    return model(x, state)
            cases["forward_%s_input_%s" % (fmt, "fp32" if inp == "fp32" else "half")] = (fwd, None)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        return e0, e1

    for _ in range(args.warmup):
        for fn, _ in cases.values():
            timed(fn)
    torch.cuda.synchronize()
    ms = {k: [] for k in cases}
    for rep in range(args.reps):
        order = list(cases) if rep % 2 == 0 else list(reversed(list(cases)))  # alternate the order too
        evs = {k: timed(cases[k][0]) for k in order}
        torch.cuda.synchronize()
        for k, (a, b) in evs.items():
            ms[k].append(a.elapsed_time(b))
    res = {}
    for k, (_, nbytes) in cases.items():
        v = ms[k]
        r = dict(ms=round(statistics.median(v), 4), ms_min=round(min(v), 4), ms_max=round(max(v), 4), n=len(v))
        if nbytes:
            r["obs_bytes_per_s"] = round(nbytes / (r["ms"] * 1e-3) / 1e9, 1) * 1e9
        res[k] = r
    for layout in shape:
        for path in rows:
            base = res["observe_%s_fp32_%s" % (layout, path)]["ms"]
            for fmt in FORMATS:
                res["observe_%s_%s_%s" % (layout, fmt, path)]["vs_fp32"] = round(
                    res["observe_%s_%s_%s" % (layout, fmt, path)]["ms"] / base, 4)
        for fmt in ("fp16", "bf16"):
            c = res["cast_%s_%s_all" % (layout, fmt)]
            c["vs_fp32"] = round(c["ms"] / res["observe_%s_fp32_all" % layout]["ms"], 4)
            res["observe_%s_%s_all" % (layout, fmt)]["vs_cast"] = round(
                res["observe_%s_%s_all" % (layout, fmt)]["ms"] / c["ms"], 4)
    for fmt in ("fp16", "bf16"):
        res["forward_%s_input_half" % fmt]["vs_input_fp32"] = round(
            res["forward_%s_input_half" % fmt]["ms"] / res["forward_%s_input_fp32" % fmt]["ms"], 4)
        for inp in ("half", "fp32"):
            res["forward_%s_input_%s" % (fmt, inp)]["precision"] = "reduced (autocast %s), for scale only" % fmt
    half_all = ["observe_%s_%s_all" % (lay, f) for lay in shape for f in ("fp16", "bf16")]
    print(json.dumps(dict(
        metric="half-precision observations (SF_OBS_F16 / SF_OBS_BF16)", envs=n, setup_steps=args.setup,
        list_ids=args.list, fwd_batch=B, reps=args.reps, checked_elements=checked, outputs_equal_cast_fp32=True,
        device=torch.cuda.get_device_name(), power_limit_w=power_limit_w(), cases=res,
        goals=dict(faster_than_fp32_plus_cast=all(res[k]["vs_cast"] < 1.0 for k in half_all),
                   within_0_6_of_fp32=all(res[k]["vs_fp32"] <= 0.6 for k in half_all)))))
    sim.close()


if __name__ == "__main__":
    main()
