"""Cost of the per-agent step outputs (sf_enable_agent_out) on one GPU; writes one JSON file (--out, default
profiles/r08_agent_out.json) and prints it.

Workloads, each on two handles of the same configuration and seeds, one with agent outputs and one without, so
that both step the same arenas through the same states:
  squad-agents  Squad with the nine squad NPCs driven (10 agent slots), levels 1-10, default capacities, episodes
                truncated at 2,048 steps, auto-reset; 131,072 arenas after --setup steps
  royale16      Battle Royale, 16 players in 4 teams, max_steps 2,048, auto-reset (bench.py --workload royale16);
                32,768 arenas after --setup steps
The actions are the 28-symbol synthetic stream (the same row for both handles).

Cases, each one call timed with CUDA events around it, alternating on / off and rotating the order from one
repetition to the next (--reps after --warmup; medians):
  step_off      sf_step of the handle without agent outputs
  step_on       sf_step of the handle with agent outputs (the AGENTS kernel)
  get           sf_get(SF_FIELD_AGENT_OUT) into a preallocated buffer
The state hashes of the two handles are compared after the run.  The card name, its power limit and its SM clock
are read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from strikeforce_b200 import config as sfcfg  # noqa: E402
from strikeforce_b200.lib import lib  # noqa: E402
from strikeforce_b200.sim import BatchedArena  # noqa: E402

WORKLOADS = {
    "squad-agents": (131072, dict(mode="Squad", level=1, level_max=10, squad_agents=True, max_steps=2048, auto_reset=True)),
    "royale16": (32768, dict(mode="Royale", teams=[1, 2, 3, 4] * 4, max_steps=2048, auto_reset=True)),
}


def smi(field):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=" + field,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
        return out.strip().splitlines()[0]
    except Exception:  # no nvidia-smi on the host: the value is reported as unknown
        return None


def run(name, n, kw, args):
    on, off = BatchedArena(n, agent_out=True, **kw), BatchedArena(n, **kw)
    table = sfcfg.ACTIONS28
    for t in range(args.setup):
        act = on.synth_actions(t, table)
        on.step(act)
        off.step(act)
    t = args.setup
    rows = torch.empty((n, on.n_agents, 5), dtype=torch.int32, device=on.device)
    stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
    get = lambda: lib().sf_get(on._h, sfcfg.FIELD_AGENT_OUT, C.c_void_p(rows.data_ptr()), stream())  # noqa: E731
    names = ["step_off", "step_on", "get"]
    ms = {c: [] for c in names}
    acts = []
    for r in range(args.warmup + args.reps):
        act = on.synth_actions(t + r, table).clone()
        acts.append(act)
        cases = {"step_off": lambda: off.step(act), "step_on": lambda: on.step(act), "get": get}
        order = names[:2] if r % 2 == 0 else names[1::-1]
        for c in order + ["get"]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            assert cases[c]() in (None, 0)
            e1.record()
            e1.synchronize()
            if r >= args.warmup:
                ms[c].append(e0.elapsed_time(e1))
    assert torch.equal(on.state_hash(), off.state_hash()), "%s: the two handles' states differ" % name
    assert torch.equal(on.step_out(), off.step_out())
    flags = rows[:, :, 0]
    res = {c: dict(ms=round(statistics.median(v), 4), ms_min=round(min(v), 4), ms_max=round(max(v), 4), n=len(v))
           for c, v in ms.items()}
    ratio = res["step_on"]["ms"] / res["step_off"]["ms"]
    out = dict(envs=n, agents_per_env=on.n_agents, setup_steps=args.setup, cases=res,
               step_on_over_off=round(ratio, 4), get_over_step_off=round(res["get"]["ms"] / res["step_off"]["ms"], 4),
               rows_last_step=dict(driven=int(((flags & sfcfg.AGENT_DRIVEN) != 0).sum()),
                                   died=int(((flags & sfcfg.AGENT_DIED) != 0).sum()),
                                   kills=int((rows[:, :, 4] != 0).sum())),
               goal_at_most_1_05x=bool(ratio <= 1.05))
    on.close(), off.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", default="squad-agents,royale16")
    ap.add_argument("--envs", type=int, default=0, help="arenas per workload (0: the defaults above)")
    ap.add_argument("--setup", type=int, default=1024, help="steps before the measurement")
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_agent_out.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_agent_out.py measures the GPU kernels; no CUDA device is usable")
    res = {}
    for name in args.workloads.split(","):
        n, kw = WORKLOADS[name]
        res[name] = run(name, args.envs or n, kw, args)
    out = dict(metric="sf_step with agent outputs against without, same arenas", device=torch.cuda.get_device_name(),
               power_limit_w=smi("power.limit"), sm_clock_mhz=smi("clocks.sm"), reps=args.reps, workloads=res)
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
