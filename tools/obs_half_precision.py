"""What fp16 and bfloat16 do to the observation values of the test workloads, computed on the CPU from the C
oracle's fp32 observations (no GPU); prints one JSON line.

Workloads: the configurations of tests/test_gpu_obs_half.py -- Squad with agents, Solo (levels 1-10, one arena
per level) and 16-player Royale (--royale arenas) -- on the synthetic 28-symbol action stream with auto-reset,
every observable slot observed every --every steps for --steps steps.  For each format: the distinct non-zero
fp32 values seen, and how many of them share their converted value with another of them (round to nearest even,
as SF_OBS_F16 / SF_OBS_BF16 write them)."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import common  # noqa: E402
import sfo  # noqa: E402
from strikeforce_b200 import config as sfcfg  # noqa: E402
from strikeforce_b200 import data as sfdata  # noqa: E402
from test_split_step import ROYALE_CAPS, SMALL, SQUAD_CAPS  # noqa: E402


def collect(arena, mode, levels, steps, every, **kw):
    vals = set()
    for i, lvl in enumerate(levels):
        cfg = sfcfg.make_config(arena, mode=mode, level_min=lvl, **kw)
        o = sfo.Arena(cfg)
        o.reset(lvl, common.synth_tb(i), common.synth_serial(i, 0))
        for t in range(steps):
            o.step(bytes(common.synth_actions([i], sfcfg.MAX_PLAYERS, t, sfcfg.ACTIONS28)[0]))
            if o.status() != sfcfg.RUNNING:
                o.reset(lvl, common.synth_tb(i), common.synth_serial(i, t + 1))
            if t % every:
                continue
            for slot in range(sfcfg.MAX_PLAYERS):
                try:
                    x = o.observe(slot)
                except RuntimeError:
                    continue
                vals.update(np.unique(x[x != 0]).tolist())
    return vals


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--every", type=int, default=10)
    ap.add_argument("--royale", type=int, default=3)
    args = ap.parse_args()
    arena = sfdata.load_default()
    vals = set()
    vals |= collect(arena, sfcfg.MODE_SQUAD, range(1, 11), args.steps, args.every, squad_agents=True, caps=SQUAD_CAPS)
    vals |= collect(arena, sfcfg.MODE_SOLO, range(1, 11), args.steps, args.every, caps=SMALL)
    vals |= collect(arena, sfcfg.MODE_ROYALE, [1] * args.royale, args.steps, args.every, teams=[1, 2, 3, 4] * 4,
                    caps=ROYALE_CAPS)
    v = torch.tensor(sorted(vals), dtype=torch.float32)
    res = dict(distinct_nonzero=len(vals), min=float(v.min()), max=float(v.max()))
    for name, dt in (("fp16", torch.float16), ("bf16", torch.bfloat16)):
        _, counts = torch.unique(v.to(dt).view(torch.int16), return_counts=True)
        res[name] = dict(distinct_after=int(counts.numel()), sharing=int(counts[counts > 1].sum()))
    print(json.dumps(dict(metric="observation values under fp16 / bf16 (C oracle, CPU)", steps=args.steps,
                          every=args.every, **res)))


if __name__ == "__main__":
    main()
