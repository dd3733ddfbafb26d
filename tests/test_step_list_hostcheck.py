"""sf_step_list on the host-check build of the device tick: stepping a subset S of the arenas and then its
complement must leave every arena, its sf_step_out, the statistics and the arena records exactly as one sf_step of
all arenas does, and stepping S must leave every arena outside S untouched.  The configurations and small
capacities are those of test_split_step.py, so that many episodes end, some of them in an abort.  Without
auto-reset both simulators reset their finished arenas after every step.  The GPU tests
(test_gpu_step_list.py) repeat this through the real kernels."""
import numpy as np
import pytest

import common
import listcheck
from strikeforce_b200 import config as sfcfg
from test_split_step import BASE, CONFIGS, MAX_STEPS, N

STEPS = 300
IDLE = ord("_")


def _lists(rng, n_agents, act):
    """a random subset S of the arenas and its complement as two (ids, rows) lists: S in random order, with repeated
    ids carrying all-'_' rows at higher indices and out-of-range ids, which must be skipped"""
    inside = rng.random(N) < rng.random()
    out = []
    for part in (np.nonzero(inside)[0], np.nonzero(~inside)[0]):
        ids = rng.permutation(part)
        rows = act[ids]
        if len(ids):
            dup = rng.choice(ids, size=rng.integers(1, 4))
            bad = np.array([-1, N, 1 << 30, -(1 << 31)])[:rng.integers(0, 5)]
            ids = np.concatenate([ids, dup, bad])
            rows = np.concatenate([rows, np.full((len(dup), n_agents), IDLE, np.uint8),
                                   act[rng.integers(0, N, len(bad))]])
        out.append((part, ids.astype(np.int32), rows))
    return out


def _snapshot(sim):
    return [sim.state_hash(e) for e in range(N)], [sim.step_out(e) for e in range(N)]


@pytest.mark.parametrize("auto_reset", [True, False], ids=["auto-reset", "reset-finished"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_step_list_in_two_parts_equals_step(arena_data, name, auto_reset):
    """Two host simulators on the same seeds and actions.  Every step the reference takes one hc_step of all arenas;
    the other takes hc_step_list of a random subset S (random order, repeated ids with '_' rows above their first
    entry, out-of-range ids) and then of the complement.  After S: the arenas in S equal the reference's, every other
    arena keeps its state hash and sf_step_out.  After the complement: every state hash and sf_step_out equals the
    reference's, and the statistics do.  At the end the hc_save records are equal byte for byte."""
    kw, extra = CONFIGS[name]
    cfg = sfcfg.make_config(arena_data, n_envs=N, auto_reset=auto_reset, max_steps=MAX_STEPS, env_id_base=BASE, **kw)
    ref, sim = listcheck.ListSim(cfg, extra=extra), listcheck.ListSim(cfg, extra=extra)
    rng = np.random.default_rng(sum(map(ord, name)) + auto_reset)
    ends = partial = 0
    for t in range(STEPS):
        act = common.synth_actions(range(BASE, BASE + N), ref.n_agents, t, sfcfg.ACTIONS28)
        ref.step(act.tobytes())
        (s_part, s_ids, s_rows), (c_part, c_ids, c_rows) = _lists(rng, ref.n_agents, act)
        hashes, outs = _snapshot(sim)
        sim.step_list(s_rows, s_ids)
        inside = set(s_part.tolist())
        partial += 0 < len(inside) < N
        for e in range(N):
            if e in inside:
                assert sim.state_hash(e) == ref.state_hash(e), "state in S: step %d arena %d" % (t, e)
                assert sim.step_out(e) == ref.step_out(e), "step_out in S: step %d arena %d" % (t, e)
            else:
                assert sim.state_hash(e) == hashes[e], "state outside S changed: step %d arena %d" % (t, e)
                assert sim.step_out(e) == outs[e], "step_out outside S changed: step %d arena %d" % (t, e)
        sim.step_list(c_rows, c_ids)
        for e in range(N):
            assert sim.step_out(e) == ref.step_out(e), "step_out: step %d arena %d" % (t, e)
            assert sim.state_hash(e) == ref.state_hash(e), "state: step %d arena %d" % (t, e)
            ends += ref.step_out(e)["status"] != sfcfg.RUNNING
        assert sim.stats() == ref.stats(), "statistics: step %d" % t
        if not auto_reset:
            ref.reset_finished()
            sim.reset_finished()
    for e in range(N):
        a, b = ref.save(e), sim.save(e)
        assert (a == b).all(), "record of arena %d differs at bytes %s" % (e, np.nonzero(a != b)[0][:16])
    assert ends >= 2 * N, "only %d episodes ended" % ends
    assert partial >= STEPS // 2


def test_step_list_skips_repeats_and_bad_ids(arena_data):
    """A list of nothing but out-of-range ids, and the empty list, change nothing and count nothing; an id listed
    twice is stepped once, with the row of its first entry: the later entry's '_' row is not applied and the arena
    is not stepped a second time."""
    kw, extra = CONFIGS["squad-agents"]
    cfg = sfcfg.make_config(arena_data, n_envs=N, auto_reset=True, max_steps=MAX_STEPS, env_id_base=BASE, **kw)
    ref, sim = listcheck.ListSim(cfg, extra=extra), listcheck.ListSim(cfg, extra=extra)
    na = ref.n_agents
    for t in range(40):
        act = common.synth_actions(range(BASE, BASE + N), na, t, sfcfg.ACTIONS28)
        ref.step(act.tobytes())
        sim.step(act.tobytes())
    stats, (hashes, outs) = sim.stats(), _snapshot(sim)
    sim.step_list(np.zeros((4, na), np.uint8) + IDLE, [-1, N, N + 5, -(1 << 31)])
    sim.step_list(np.zeros((0, na), np.uint8), [])
    assert sim.stats() == stats and _snapshot(sim) == (hashes, outs)
    act = common.synth_actions(range(BASE, BASE + N), na, 40, sfcfg.ACTIONS28)
    assert (act[3] != IDLE).any()
    ref.step(act.tobytes())
    ids = np.array([3] + [e for e in range(N) if e != 3] + [3, 3], np.int32)
    rows = np.concatenate([act[ids[:N]], np.full((2, na), IDLE, np.uint8)])
    sim.step_list(rows, ids)
    assert _snapshot(sim) == _snapshot(ref)
    assert sim.stats() == ref.stats()
