"""sf_reset_finished / sf_list_finished on the host-check build of the device tick: auto_reset = 0 plus a reset
of the finished arenas right after every step must leave every arena, its sf_step_out, the statistics and the
arena records exactly as auto_reset = 1 does, with the full step and with the split step.  Between the step and
the reset the terminal state can be observed; it must be what the C oracle shows for its terminal state.  The
configurations and small capacities are those of test_split_step.py, so that many episodes end, some of them
inside half A.  The GPU tests (test_gpu_reset_finished.py) repeat this through the real kernels."""
import numpy as np
import pytest

import common
import finishcheck
import sfo
from strikeforce_b200 import config as sfcfg
from test_split_step import ABORTS, BASE, CONFIGS, MAX_STEPS, N, STEPS, _level

ENDS = (sfcfg.WIN, sfcfg.DEAD, sfcfg.TIMEOUT, sfcfg.TRUNCATED)


def _pair(arena_data, name):
    kw, extra = CONFIGS[name]
    return [finishcheck.FinishSim(sfcfg.make_config(arena_data, n_envs=N, auto_reset=ar, max_steps=MAX_STEPS,
                                                    env_id_base=BASE, **kw), extra=extra) for ar in (True, False)]


def _step(sim, act, split):
    if split:
        sim.step(None, half=1)
        sim.step(act, half=2)
    else:
        sim.step(act)


@pytest.mark.parametrize("split", [False, True], ids=["full-step", "split-step"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_reset_finished_equals_auto_reset(arena_data, name, split):
    """Two host simulators on the same seeds and actions: one with auto-reset, one without it and
    hc_reset_finished after every step.  hc_list_finished before the reset is the ascending list of the arenas
    whose step ended the episode, and empty after it; sf_step_out and the state hash of every arena after every
    step, the statistics and the hc_save record of every arena at the end are equal."""
    auto, manual = _pair(arena_data, name)
    ends = aborts = 0
    for t in range(STEPS):
        act = common.synth_actions(range(BASE, BASE + N), auto.n_agents, t, sfcfg.ACTIONS28).tobytes()
        _step(auto, act, split)
        if split:
            manual.step(None, half=1)
            aborts += sum(manual.step_out(e)["status"] in ABORTS for e in range(N))
            assert manual.list_finished().tolist() == [e for e in range(N) if manual.status(e) != sfcfg.RUNNING]
            manual.step(act, half=2)
        else:
            manual.step(act)
        ended = [e for e in range(N) if manual.step_out(e)["status"] != sfcfg.RUNNING]
        ends += len(ended)
        aborts += 0 if split else sum(manual.step_out(e)["status"] in ABORTS for e in ended)
        assert manual.list_finished().tolist() == ended, "step %d" % t
        manual.reset_finished()
        assert manual.list_finished().size == 0, "step %d" % t
        for e in range(N):
            assert manual.step_out(e) == auto.step_out(e), "step_out: step %d arena %d" % (t, e)
            assert manual.state_hash(e) == auto.state_hash(e), "state: step %d arena %d" % (t, e)
    assert manual.stats() == auto.stats()
    for e in range(N):
        a, m = auto.save(e), manual.save(e)
        assert (a == m).all(), "record of arena %d differs at bytes %s" % (e, np.nonzero(a != m)[0][:16])
    assert ends >= 2 * N, "only %d episodes ended" % ends
    assert aborts >= 15, "only %d episodes ended in an abort" % aborts


def test_reset_finished_does_nothing_with_auto_reset(arena_data):
    """With auto-reset on, no arena is ever listed and hc_reset_finished changes nothing."""
    auto, _ = _pair(arena_data, "squad-agents")
    for t in range(200):
        auto.step(common.synth_actions(range(BASE, BASE + N), auto.n_agents, t, sfcfg.ACTIONS28).tobytes())
        assert auto.list_finished().size == 0
        before = [auto.save(e) for e in range(N)]
        auto.reset_finished()
        assert all((auto.save(e) == before[e]).all() for e in range(N))


@pytest.mark.parametrize("name", list(CONFIGS))
def test_final_observation_follows_the_oracle(arena_data, name):
    """auto_reset = 0 and hc_reset_finished after every step, next to the C oracle in lock step (the oracle reset
    on the synthetic seed chain when its episode ends).  For every episode that ends in WIN / DEAD / TIMEOUT /
    TRUNCATED the observation of the terminal state, taken before the reset, equals the oracle's observation of
    its terminal state word for word: the player's slot, and every squad-agent slot for Squad with agents.  The
    state hash of every arena equals the oracle's after every reset.  With the small capacities nearly every
    episode ends in an overflow, whose terminal state is undefined, so this test runs at the default ones, where
    the episodes end at max_steps (TRUNCATED)."""
    kw, extra = CONFIGS[name]
    kw = {key: v for key, v in kw.items() if key != "caps"}
    hs = finishcheck.FinishSim(sfcfg.make_config(arena_data, n_envs=N, auto_reset=False, max_steps=MAX_STEPS,
                                                 env_id_base=BASE, **kw), extra=extra)
    okw = {key: v for key, v in kw.items() if key not in ("level_min", "level_max")}
    oracles = []
    for e in range(N):
        o = sfo.Arena(sfcfg.make_config(arena_data, level_min=_level(kw, e), max_steps=MAX_STEPS, **okw))
        o.reset(_level(kw, e), common.synth_tb(BASE + e), common.synth_serial(BASE + e, 0))
        oracles.append(o)
    slots = range(hs.n_agents) if kw.get("squad_agents") else [0]
    episode = [0] * N
    compared = ends = 0
    for t in range(STEPS):
        act = common.synth_actions(range(BASE, BASE + N), hs.n_agents, t, sfcfg.ACTIONS28)
        hs.step(act.tobytes())
        sts = [o.step(bytes(act[e])) for e, o in enumerate(oracles)]
        assert hs.list_finished().tolist() == [e for e in range(N) if sts[e] != sfcfg.RUNNING], "step %d" % t
        for e, o in enumerate(oracles):
            assert hs.step_out(e)["status"] == sts[e], "status: step %d arena %d" % (t, e)
            if sts[e] not in ENDS:
                continue
            ends += 1
            for slot in slots:
                try:
                    ref = o.observe(slot)
                except RuntimeError:
                    continue  # no agent in that slot any more
                got = hs.observe(e, slot)
                assert (got.view(np.uint32) == ref.view(np.uint32)).all(), \
                    "terminal observation: step %d arena %d slot %d" % (t, e, slot)
                compared += 1
        hs.reset_finished()
        for e, o in enumerate(oracles):
            if sts[e] != sfcfg.RUNNING:
                episode[e] += 1
                o.reset(_level(kw, e), common.synth_tb(BASE + e), common.synth_serial(BASE + e, episode[e]))
            assert np.uint64(hs.state_hash(e)) == np.uint64(o.state_hash()), "state: step %d arena %d" % (t, e)
    assert ends >= N, "only %d episodes ended in WIN / DEAD / TIMEOUT / TRUNCATED" % ends
    assert compared >= ends, "only %d terminal observations compared" % compared
