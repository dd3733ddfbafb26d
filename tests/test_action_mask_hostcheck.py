"""sf_action_mask on the host-check build of the device code: the predicate the CUDA kernel runs
(hc_action_mask) must equal the definition of the mask applied literally (hc_action_mask_brute: obey every
delivered symbol on a saved copy of the arena, compare its canonical hash and status with those after '+',
restore the record), at P1 and at P2, along trajectories of the 28-symbol stream with the synthetic player sheet
(it owns every item, so selections, throws, shots, blocks and portals all occur) and small capacities (so a
command can overflow an arena).  Also on the spill-stress build of the flag table and on the 3x40x128 map.  The
GPU tests (test_gpu_action_mask.py) compare the CUDA kernel with the brute force."""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.dirname(HERE), os.path.join(os.path.dirname(HERE), "oracle"), HERE, os.path.join(HERE, "hostcheck")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import common  # noqa: E402
import maskcheck  # noqa: E402
from strikeforce_b200 import config as sfcfg  # noqa: E402
from strikeforce_b200 import data as sfdata  # noqa: E402
from test_split_step import ROYALE_CAPS, SMALL, SQUAD_CAPS  # noqa: E402

SPILL_STRESS = ("-DSF_BT_SLOTS=7", "-DSF_BT_FULL=5")  # as in test_hostcheck.py: the flag table spills constantly
SYN = dict(player="synthetic")
# name -> (make_config keywords, compiler flags of the host build)
CONFIGS = {
    "solo": (dict(mode=sfcfg.MODE_SOLO, level_min=1, level_max=10, caps=SMALL, **SYN), ()),
    "timer": (dict(mode=sfcfg.MODE_TIMER, level_min=1, level_max=10, caps=SMALL, **SYN), ()),
    "squad": (dict(mode=sfcfg.MODE_SQUAD, level_min=1, level_max=10, caps=SQUAD_CAPS, **SYN), ()),
    "squad-agents": (dict(mode=sfcfg.MODE_SQUAD, level_min=1, level_max=10, squad_agents=True, caps=SQUAD_CAPS, **SYN),
                     ()),
    "squad-agents-tiny-flag-table": (dict(mode=sfcfg.MODE_SQUAD, level_min=1, level_max=10, squad_agents=True,
                                          caps=SQUAD_CAPS, **SYN), SPILL_STRESS),
    "royale16-ind5": (dict(mode=sfcfg.MODE_ROYALE, teams=[1, 2, 3, 4] * 4, caps=ROYALE_CAPS, ind=5, **SYN), ()),
}
N, STEPS, EVERY, BASE, MAX_STEPS = 8, 60, 3, 300, 45  # a truncation lands on a checked step
AGENT_BITS = sum(1 << sfcfg.COMMANDS.index(c) for c in b"+xzqeawsd")
ALWAYS = b"+qe"  # '+' by rule; a turn always changes the facing
NEVER = b"3"     # obey ignores it


def run(name, arena, n=N, steps=STEPS):
    """Steps a MaskSim of config `name`; at P1 and P2 of every EVERY-th step the predicate equals the brute force.
    Returns the bits seen set and clear on controllable slots."""
    kw, extra = CONFIGS[name]
    # no auto-reset: an arena that ended stays finished until after its P1 mask (sf_reset_finished then)
    cfg = sfcfg.make_config(arena, n_envs=n, auto_reset=False, max_steps=MAX_STEPS, env_id_base=BASE, **kw)
    sim = maskcheck.MaskSim(cfg, extra=maskcheck.EXTRA + extra)  # EXTRA: the geometry of SF_GEOMETRY
    seen_set = seen_clear = 0
    agent_slots = finished = 0
    for t in range(steps):
        act = common.synth_actions(range(BASE, BASE + n), sim.n_agents, t, sfcfg.ACTIONS28).tobytes()
        for half, point in ((1, "P1"), (2, "P2")):
            if t % EVERY == 0:
                got, want = sim.masks(), sim.masks(brute=True)
                bad = np.argwhere(got != want)
                assert not len(bad), "%s step %d %s: arena %d slot %d: %s vs brute force %s" % (
                    name, t, point, bad[0][0], bad[0][1], bin(got[tuple(bad[0])]), bin(want[tuple(bad[0])]))
                assert not (got >> sfcfg.N_COMMANDS).any()
                for e in range(n):
                    if sim.status(e) != sfcfg.RUNNING:
                        assert not got[e].any(), "finished arena %d has a mask" % e
                        finished += 1
                for m in got[got != 0]:
                    assert m & 1, "a controllable slot without '+'"
                    seen_set |= int(m)
                    seen_clear |= ~int(m) & ((1 << sfcfg.N_COMMANDS) - 1)
                if kw["mode"] == sfcfg.MODE_SQUAD:  # slots above 0 are squad agents (or nothing)
                    assert not (got[:, 1:] & ~np.uint32(AGENT_BITS)).any(), "a squad agent with a bit outside +xzqeawsd"
                    agent_slots += int((got[:, 1:] != 0).sum())
            if half == 1:
                sim.reset_finished()
            sim.step(None if half == 1 else act, half=half)
    if kw.get("squad_agents"):
        assert agent_slots > 0
    return seen_set, seen_clear, finished


def test_commands_mirror_the_header():
    assert sfcfg.COMMANDS == maskcheck.commands()
    assert len(sfcfg.COMMANDS) == sfcfg.N_COMMANDS == 30 and sfcfg.COMMANDS[:-1].replace(b"3", b"") == sfcfg.ACTIONS28


@pytest.mark.parametrize("name", list(CONFIGS))
def test_mask_equals_brute_force(arena_data, name):
    seen_set, seen_clear, finished = run(name, arena_data)
    for j, c in enumerate(sfcfg.COMMANDS):
        if c in ALWAYS:
            assert (seen_set >> j) & 1 and not (seen_clear >> j) & 1, chr(c)
        elif c in NEVER:
            assert not (seen_set >> j) & 1, chr(c)
    assert finished > 0, "no finished arena was masked"


def test_every_symbol_is_seen_set_and_clear(arena_data):
    """Over the configurations: every symbol but '3' and the always-set '+', 'q', 'e' is seen set and clear on
    controllable slots ('_' is clear on squad agents)."""
    seen_set = seen_clear = 0
    for name in ("timer", "squad-agents"):
        s, c, _ = run(name, arena_data, steps=30)
        seen_set, seen_clear = seen_set | s, seen_clear | c
    for j, c in enumerate(sfcfg.COMMANDS):
        if c not in ALWAYS + NEVER:
            assert (seen_set >> j) & 1 and (seen_clear >> j) & 1, "%r is not seen both set and clear" % chr(c)


def test_mask_on_the_larger_map():
    """The 3x40x128 map: the host-check build takes the geometry from the environment, so a process of its own."""
    env = dict(os.environ, SF_GEOMETRY="40x128")
    env.pop("SF_LIB_PATH", None)
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "squad-agents", "royale16-ind5"],
                         capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert "MASK OK 40x128" in out.stdout


if __name__ == "__main__":
    arena = sfdata.load_default()
    for nm in sys.argv[1:]:
        run(nm, arena, n=4, steps=30)
    print("MASK OK %dx%d" % (sfcfg.ROWS, sfcfg.COLS))
