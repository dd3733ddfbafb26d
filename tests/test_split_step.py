"""The split step (sf_step_a, the P2 observation point, sf_step_b) on the host-check build of the device
tick: it must leave every arena, its sf_step_out and the statistics exactly as sf_step does, and follow
the C oracle driven half by half.  The capacities are small so that many episodes end inside half A
(a spawn that needs a slot beyond a capacity is SF_OVERFLOW), the case where the two paths can part:
such an arena has to keep its terminal status through half B and be reset only at the end of the step.
The GPU tests (test_gpu_launch_paths.py) repeat this through the real kernels."""
import numpy as np
import pytest

import common
import hostcheck
import sfo
from strikeforce_b200 import config as sfcfg

SPILL_STRESS = ("-DSF_BT_SLOTS=7", "-DSF_BT_FULL=5")  # as in test_hostcheck.py: the flag table spills constantly
SMALL = dict(cap_humans=12, cap_zombies=4, cap_bullets=6, cap_built=8, cap_portals=8)
SQUAD_CAPS = dict(cap_humans=12, cap_zombies=8, cap_bullets=6, cap_built=8, cap_portals=8)
ROYALE_CAPS = dict(cap_humans=20, cap_zombies=8, cap_bullets=24)

# name -> (make_config keywords, compiler flags of the host build)
CONFIGS = {
    "solo": (dict(mode=sfcfg.MODE_SOLO, level_min=1, level_max=10, caps=SMALL), ()),
    "timer": (dict(mode=sfcfg.MODE_TIMER, level_min=1, level_max=10, caps=SMALL, player="synthetic"), ()),
    "squad-agents": (dict(mode=sfcfg.MODE_SQUAD, level_min=1, level_max=10, squad_agents=True, caps=SQUAD_CAPS), ()),
    "squad-agents-tiny-flag-table": (dict(mode=sfcfg.MODE_SQUAD, level_min=1, level_max=10, squad_agents=True,
                                          caps=SQUAD_CAPS), SPILL_STRESS),
    "royale16": (dict(mode=sfcfg.MODE_ROYALE, teams=[1, 2, 3, 4] * 4, caps=ROYALE_CAPS), ()),
}
ABORTS = (sfcfg.OVERFLOW, sfcfg.UB_GUARD)
N, STEPS, BASE, MAX_STEPS = 16, 400, 300, 150


def _level(kw, e):
    lo = kw.get("level_min", 1)
    return lo + (BASE + e) % (kw.get("level_max", lo) - lo + 1)


@pytest.mark.parametrize("auto_reset", [True, False], ids=["auto-reset", "harness-reset"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_split_step_equals_full_step(arena_data, name, auto_reset):
    """Two host simulators on the same seeds and actions, one stepped with sf_step and one with
    sf_step_a + sf_step_b: state hash and sf_step_out of every arena after every step, the statistics at
    the end.  Without auto-reset the test resets ended episodes itself, on the synthetic seed chain."""
    kw, extra = CONFIGS[name]
    cfg = sfcfg.make_config(arena_data, n_envs=N, auto_reset=auto_reset, max_steps=MAX_STEPS, env_id_base=BASE, **kw)
    full, split = hostcheck.HostSim(cfg, extra=extra), hostcheck.HostSim(cfg, extra=extra)
    episode = [0] * N
    aborts_in_a = 0
    for t in range(STEPS):
        act = common.synth_actions(range(BASE, BASE + N), full.n_agents, t, sfcfg.ACTIONS28).tobytes()
        live = [split.status(e) == sfcfg.RUNNING for e in range(N)]
        full.step(act)
        split.step(None, half=1)
        aborts_in_a += sum(live[e] and split.step_out(e)["status"] in ABORTS for e in range(N))
        split.step(act, half=2)
        for e in range(N):
            assert split.step_out(e) == full.step_out(e), "step_out: step %d arena %d" % (t, e)
            assert split.state_hash(e) == full.state_hash(e), "state: step %d arena %d" % (t, e)
            if full.step_out(e)["status"] != sfcfg.RUNNING:
                episode[e] += 1
                if not auto_reset:
                    for hs in (full, split):
                        hs.reset(e, common.synth_tb(BASE + e), common.synth_serial(BASE + e, episode[e]))
    assert split.stats() == full.stats()
    st = full.stats()
    assert st["episodes"] == sum(episode)
    assert st["steps"] + st["overflows"] + st["ub_guards"] == N * STEPS
    assert aborts_in_a >= 15, "only %d episodes ended inside half A" % aborts_in_a


@pytest.mark.parametrize("auto_reset", [True, False], ids=["auto-reset", "harness-reset"])
def test_split_step_follows_the_oracle(arena_data, auto_reset):
    """Squad with agent-driven squad humans, stepped half by half next to the C oracle (sfo_step_a /
    sfo_step_b, the oracle reset on the synthetic seed chain when an episode ends): status every step,
    the whole sf_step_out of every step that ran to its end, the state hash after every step, and the
    P2 observations of all squad-agent slots bit for bit.  An arena that ended in half A has no
    defined P2 observation and is skipped, as is a slot whose human is gone."""
    kw, _ = CONFIGS["squad-agents"]
    cfg = sfcfg.make_config(arena_data, n_envs=N, auto_reset=auto_reset, max_steps=MAX_STEPS, env_id_base=BASE, **kw)
    hs = hostcheck.HostSim(cfg)
    oracles = []
    for e in range(N):
        lvl = _level(kw, e)
        o = sfo.Arena(sfcfg.make_config(arena_data, mode=kw["mode"], level_min=lvl, squad_agents=True, caps=kw["caps"],
                                        max_steps=MAX_STEPS))
        o.reset(lvl, common.synth_tb(BASE + e), common.synth_serial(BASE + e, 0))
        oracles.append(o)
    episode = [0] * N
    aborts_in_a = compared = 0
    for t in range(STEPS):
        act = common.synth_actions(range(BASE, BASE + N), hs.n_agents, t, sfcfg.ACTIONS28)
        hs.step(None, half=1)
        ended_in_a = [o.step_a() != sfcfg.RUNNING for o in oracles]
        aborts_in_a += sum(ended_in_a)
        for e, o in enumerate(oracles):
            assert hs.step_out(e)["status"] == o.status(), "status after half A: step %d arena %d" % (t, e)
            if ended_in_a[e] or t % 4:
                continue
            for slot in range(1, hs.n_agents):
                try:
                    ref = o.observe(slot)
                except RuntimeError:
                    continue  # that human is gone: its agent builds nothing
                got = hs.observe(e, slot)
                assert (got.view(np.uint32) == ref.view(np.uint32)).all(), "P2 observation: step %d arena %d slot %d" % (t, e, slot)
                compared += 1
        hs.step(act.tobytes(), half=2)
        for e, o in enumerate(oracles):
            st = o.step_b(bytes(act[e])) if not ended_in_a[e] else o.status()
            out = hs.step_out(e)
            assert out["status"] == st, "status: step %d arena %d" % (t, e)
            if st not in ABORTS:
                assert out == o.step_out(), "step_out: step %d arena %d" % (t, e)
            if st != sfcfg.RUNNING:
                episode[e] += 1
                tb, serial = common.synth_tb(BASE + e), common.synth_serial(BASE + e, episode[e])
                o.reset(_level(kw, e), tb, serial)
                if not auto_reset:
                    hs.reset(e, tb, serial)
            assert np.uint64(hs.state_hash(e)) == np.uint64(o.state_hash()), "state: step %d arena %d" % (t, e)
    st = hs.stats()
    assert st["episodes"] == sum(episode)
    assert st["steps"] + st["overflows"] + st["ub_guards"] == N * STEPS
    assert aborts_in_a >= 15, "only %d episodes ended inside half A" % aborts_in_a
    assert compared >= 1000
