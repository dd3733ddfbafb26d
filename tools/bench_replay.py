"""Cost of replay (sf_enable_replay / sf_replay_load) on one GPU; writes one JSON file (--out, default
profiles/r10_replay.json) and prints it.

Workloads (those of tools/bench_match_log.py):
  squad-agents  Squad with the nine squad NPCs driven (10 agent slots), levels 1-10, default capacities, episodes
                truncated at 2,048 steps, auto-reset; 131,072 arenas
  royale16      Battle Royale, 16 players in 4 teams, max_steps 2,048, auto-reset; 32,768 arenas
The actions are the 28-symbol synthetic stream (the same row for every handle).

First a recording handle with match logs and no auto-reset plays --setup + --warmup + --reps steps from the first
reset and exports every arena's tape: its first episode, or as much of it as was played.  Then four fresh handles
of the same configuration -- one with replay and every tape loaded, one with match logs, one with agent outputs, one
with none of these -- play the same steps: the replay handle deals the recorded commands, which are the commands the
others are given, so all four step the same arenas through the same states (an arena whose tape ended follows the
action rows, as the others do).

Two windows of --reps steps after --warmup ones, each step one call timed with CUDA events around it, the four
handles in an order rotated from one repetition to the next (medians):
  steady  after --setup steps from the load: mid-episode populations, but only the arenas whose first episode is
          still running have an armed tape (most squad-agents arenas, few royale16 ones)
  fresh   then every handle is put back at the start (the replay handle by loading the tapes again, the others by
          sf_reset with the same seeds) and the first steps of the tapes are timed: every tape armed
Cases in each window:
  step_off      sf_step of the handle with none of the extras
  step_replay   sf_step of the replay handle (the EXTRAS kernel dealing from the armed tapes)
  step_log      sf_step of the handle with match logs
  step_agent    sf_step of the handle with agent outputs
and load, sf_replay_load of every arena (timed on the replay handle before its steps: each load resets the arenas to
the same start).  The state hashes and step outputs of the four handles are compared after each window, and the
share of arenas whose tape is still armed is reported.  The card name, its power limit and its SM clock are read in
the same run."""
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


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def run(name, n, kw, args):
    table = sfcfg.ACTIONS28
    total = args.setup + args.warmup + args.reps
    probe = BatchedArena(32, **kw)
    cap = probe.n_agents * kw["max_steps"]
    probe.close()
    rec = BatchedArena(n, match_log=cap, **dict(kw, auto_reset=False))
    for t in range(total):
        rec.step(rec.synth_actions(t, table))
    rows = rec.match_logs()
    rec.close()
    ids = torch.arange(n, dtype=torch.int32, device=rows.device)
    rp = BatchedArena(n, replay=cap, **kw)
    load_ms = []
    for r in range(args.warmup + args.reps):
        ms = timed(lambda: rp.replay_load(rows, ids))
        if r >= args.warmup:
            load_ms.append(ms)
    status = rp.replay_load(rows, ids)
    assert int(status.item()) == 0, "%s: tapes refused" % name
    log, agent, off = BatchedArena(n, match_log=cap, **kw), BatchedArena(n, agent_out=True, **kw), BatchedArena(n, **kw)
    handles = dict(step_replay=rp, step_log=log, step_agent=agent, step_off=off)
    names = list(handles)

    def window(t0):
        ms = {c: [] for c in names}
        for r in range(args.warmup + args.reps):
            act = off.synth_actions(t0 + r, table).clone()
            k = r % len(names)
            for c in names[k:] + names[:k]:
                v = timed(lambda: handles[c].step(act))
                if r >= args.warmup:
                    ms[c].append(v)
        for h in (rp, log, agent):
            assert torch.equal(h.state_hash(), off.state_hash()), "%s: the handles' states differ" % name
            assert torch.equal(h.step_out(), off.step_out())
        state = rp.replay_state()
        res = {c: dict(ms=round(statistics.median(v), 4), ms_min=round(min(v), 4), ms_max=round(max(v), 4), n=len(v))
               for c, v in ms.items()}
        ratio = res["step_replay"]["ms"] / res["step_off"]["ms"]
        return dict(cases=res, step_replay_over_off=round(ratio, 4),
                    step_log_over_off=round(res["step_log"]["ms"] / res["step_off"]["ms"], 4),
                    step_agent_over_off=round(res["step_agent"]["ms"] / res["step_off"]["ms"], 4),
                    armed_at_end=round(float((state[:, 0] & sfcfg.REPLAY_ARMED != 0).float().mean()), 4),
                    surplus=int((state[:, 0] & sfcfg.REPLAY_SURPLUS != 0).sum()))

    for t in range(args.setup):
        act = off.synth_actions(t, table)
        for h in handles.values():
            h.step(act)
    steady = window(args.setup)
    assert int(rp.replay_load(rows, ids).item()) == 0
    for h in (log, agent, off):
        h.reset()
    fresh = window(0)
    load = dict(ms=round(statistics.median(load_ms), 4), ms_min=round(min(load_ms), 4), ms_max=round(max(load_ms), 4),
                n=len(load_ms))
    out = dict(envs=n, agents_per_env=off.n_agents, cap_symbols=cap, setup_steps=args.setup, load=load,
               steady=steady, fresh=fresh, goal_at_most_1_05x=bool(fresh["step_replay_over_off"] <= 1.05))
    for h in handles.values():
        h.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", default="squad-agents,royale16")
    ap.add_argument("--envs", type=int, default=0, help="arenas per workload (0: the defaults above)")
    ap.add_argument("--setup", type=int, default=1024, help="steps before the measurement")
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_replay.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_replay.py measures the GPU kernels; no CUDA device is usable")
    res = {}
    for name in args.workloads.split(","):
        n, kw = WORKLOADS[name]
        res[name] = run(name, args.envs or n, kw, args)
    out = dict(metric="sf_step with every replay tape armed against without, same arenas",
               device=torch.cuda.get_device_name(), power_limit_w=smi("power.limit"), sm_clock_mhz=smi("clocks.sm"),
               reps=args.reps, workloads=res)
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
