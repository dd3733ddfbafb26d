"""Cost of the match logs (sf_enable_log / sf_log_list) on one GPU; writes one JSON file (--out, default
profiles/r09_match_log.json) and prints it.

Workloads, each on three handles of the same configuration and seeds -- one with match logs, one with agent
outputs, one with neither -- so that all step the same arenas through the same states:
  squad-agents  Squad with the nine squad NPCs driven (10 agent slots), levels 1-10, default capacities, episodes
                truncated at 2,048 steps, auto-reset; 131,072 arenas after --setup steps
  royale16      Battle Royale, 16 players in 4 teams, max_steps 2,048, auto-reset (bench.py --workload royale16);
                32,768 arenas after --setup steps
The tapes hold agents_per_env * 2,048 symbols, a whole episode.  The actions are the 28-symbol synthetic stream (the
same row for every handle).

Cases, each one call timed with CUDA events around it, the three steps in an order rotated from one repetition to
the next (--reps after --warmup; medians):
  step_off      sf_step of the handle with neither
  step_log      sf_step of the handle with match logs (the EXTRAS kernel, agent-output guard not taken)
  step_agent    sf_step of the handle with agent outputs (the EXTRAS kernel, log guards not taken)
  export        sf_log_list of every arena into a preallocated buffer
The state hashes and step outputs of the three handles are compared after the run.  The card name, its power limit
and its SM clock are read in the same run."""
import argparse
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
    probe = BatchedArena(32, **kw)
    cap = probe.n_agents * kw["max_steps"]
    probe.close()
    log, agent, off = BatchedArena(n, match_log=cap, **kw), BatchedArena(n, agent_out=True, **kw), BatchedArena(n, **kw)
    handles = dict(step_log=log, step_agent=agent, step_off=off)
    table = sfcfg.ACTIONS28
    for t in range(args.setup):
        act = off.synth_actions(t, table)
        for h in handles.values():
            h.step(act)
    t = args.setup
    rows = torch.empty((n, lib().sf_log_row_bytes(log._h)), dtype=torch.uint8, device=log.device)
    names = list(handles)
    ms = {c: [] for c in names + ["export"]}
    for r in range(args.warmup + args.reps):
        act = off.synth_actions(t + r, table).clone()
        k = r % len(names)
        for c in names[k:] + names[:k] + ["export"]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if c == "export":
                log.match_logs(out=rows)
            else:
                handles[c].step(act)
            e1.record()
            e1.synchronize()
            if r >= args.warmup:
                ms[c].append(e0.elapsed_time(e1))
    for h in (log, agent):
        assert torch.equal(h.state_hash(), off.state_hash()), "%s: the handles' states differ" % name
        assert torch.equal(h.step_out(), off.step_out())
    head = rows[:, :sfcfg.LOG_HEAD.itemsize].cpu().numpy().copy().view(sfcfg.LOG_HEAD).reshape(-1)
    res = {c: dict(ms=round(statistics.median(v), 4), ms_min=round(min(v), 4), ms_max=round(max(v), 4), n=len(v))
           for c, v in ms.items()}
    ratio = res["step_log"]["ms"] / res["step_off"]["ms"]
    out = dict(envs=n, agents_per_env=off.n_agents, cap_symbols=cap, row_bytes=int(rows.shape[1]),
               setup_steps=args.setup, cases=res, step_log_over_off=round(ratio, 4),
               step_agent_over_off=round(res["step_agent"]["ms"] / res["step_off"]["ms"], 4),
               export_over_step_off=round(res["export"]["ms"] / res["step_off"]["ms"], 4),
               export_gb_per_s=round(2 * rows.numel() / res["export"]["ms"] / 1e6, 1),
               tapes=dict(complete=int((head["flags"] & sfcfg.LOG_COMPLETE != 0).sum()),
                          truncated=int((head["flags"] & sfcfg.LOG_TRUNCATED != 0).sum()),
                          mean_symbols=round(float(head["n_symbols"].mean()), 1)),
               goal_at_most_1_05x=bool(ratio <= 1.05))
    log.close(), agent.close(), off.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", default="squad-agents,royale16")
    ap.add_argument("--envs", type=int, default=0, help="arenas per workload (0: the defaults above)")
    ap.add_argument("--setup", type=int, default=1024, help="steps before the measurement")
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_match_log.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_match_log.py measures the GPU kernels; no CUDA device is usable")
    res = {}
    for name in args.workloads.split(","):
        n, kw = WORKLOADS[name]
        res[name] = run(name, args.envs or n, kw, args)
    out = dict(metric="sf_step with match logs against without, same arenas", device=torch.cuda.get_device_name(),
               power_limit_w=smi("power.limit"), sm_clock_mhz=smi("clocks.sm"), reps=args.reps, workloads=res)
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
