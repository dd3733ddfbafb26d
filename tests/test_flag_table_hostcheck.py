"""The bullet-flag table of the tick (csrc/sf_core.cuh, sf_bt_*: two-choice 4-way buckets, overflow spilled into the
overlay) on the host-check build: entry by entry against a Python set, and the rebuild from the bullet rows, which
inserts in slot order and can therefore overflow where the inserts in the order the flags were raised did not."""
import numpy as np
import pytest

import btcheck
import common
import sfo
from strikeforce_b200 import config as sfcfg
from test_hostcheck import SPILL_STRESS

FLAG_NEW, BF_SPILL, BT_SPILL = 1, 0x02000000, 0x8000


@pytest.mark.parametrize("extra", [(), SPILL_STRESS], ids=["default", "tiny"])
def test_random_inserts_lookups_and_wipes(arena_data, extra):
    """Random rounds of inserts and look-ups, each ended by a wipe, against a Python set: every answer of
    sf_flagged and sf_flag_cell, the count word, and when a flag may or must spill (never while both buckets of
    the cell can still hold it; always once SF_BT_FULL flags are in the table or, with one bucket, four)."""
    buckets, full, cells = btcheck.geometry(extra)
    sim = btcheck.BtSim(sfcfg.make_config(arena_data, n_envs=1, mode=sfcfg.MODE_SQUAD, level_min=1), extra=extra)
    rng = np.random.default_rng(7)
    env = 0
    sim.bt_wipe(env)
    spills = 0
    for rnd in range(300):
        pool = rng.choice(cells, size=int(rng.integers(4, 80)), replace=False)
        flags, spilled = set(), set()
        for _ in range(int(rng.integers(1, 160))):
            c = int(rng.choice(pool))
            if rng.random() < 0.5:
                assert sim.bt_flagged(env, c) == (c in flags), (rnd, c)
                continue
            in_table = len(flags) - len(spilled)
            fl = sim.bt_flag(env, c)
            if c in flags:
                assert fl == (BF_SPILL if c in spilled else 0), (rnd, c)
                continue
            assert fl & FLAG_NEW, (rnd, c)
            if fl & BF_SPILL:
                spilled.add(c)
                assert in_table >= min(8, 4 * buckets), "a flag spilled although its buckets had room"
            else:
                assert in_table < full and (buckets > 1 or in_table < 4), "a flag went into a full table"
            flags.add(c)
            assert sim.bt_count() == (len(flags) - len(spilled)) | (BT_SPILL if spilled else 0)
        for c in pool:
            assert sim.bt_flagged(env, int(c)) == (int(c) in flags)
        spills += len(spilled)
        sim.bt_wipe(env)
        assert sim.bt_count() == 0
        assert not any(sim.bt_flagged(env, int(c)) for c in pool)
    assert spills > 0


def test_rebuild_overflow_matches_oracle(arena_data):
    """Squad arenas followed by the C oracle every step (as the soak test of test_hostcheck.py does).  After a step,
    an arena whose flags all went into the table as they were raised, but do not all fit when the table is rebuilt
    from the bullet rows in slot order, is saved and loaded back in place, and the steps that follow, whose first
    rebuild spills, still match the oracle: state hash, sf_step_out and status.  A copy of the record shows the
    rebuild itself: the flag that did not fit is marked BF_SPILL on its bullet, and the rebuilt table answers for
    every flag."""
    n, base, max_steps = 12, 2000, 1024
    kw = dict(mode=sfcfg.MODE_SQUAD, level_min=1, level_max=10, auto_reset=True, max_steps=max_steps, env_id_base=base)
    sim = btcheck.BtSim(sfcfg.make_config(arena_data, n_envs=n, **kw))
    probe = btcheck.BtSim(sfcfg.make_config(arena_data, n_envs=1, **kw))
    oracles, episode = [], [0] * n
    for e in range(n):
        lvl = 1 + (base + e) % 10
        o = sfo.Arena(sfcfg.make_config(arena_data, mode=sfcfg.MODE_SQUAD, level_min=lvl, max_steps=max_steps))
        o.reset(lvl, common.synth_tb(base + e), common.synth_serial(base + e, 0))
        oracles.append(o)
    found = None
    for t in range(1300):
        act = common.synth_actions(range(base, base + n), 1, t, sfcfg.ACTIONS28)
        sim.step(act.tobytes())
        for e, o in enumerate(oracles):
            st = o.step(bytes(act[e]))
            assert sim.step_out(e) == o.step_out(), "step_out: step %d arena %d" % (t, e)
            if st != sfcfg.RUNNING:
                episode[e] += 1
                o.reset(1 + (base + e) % 10, common.synth_tb(base + e), common.synth_serial(base + e, episode[e]))
            assert np.uint64(sim.state_hash(e)) == np.uint64(o.state_hash()), "state: step %d arena %d" % (t, e)
        if found is not None:
            if t >= found + 8:
                break
            continue
        for e in range(n):
            cells, spilled = sim.bt_owners(e)
            if len(cells) < 8 or spilled.any() or sim.status(e) != sfcfg.RUNNING:
                continue
            rec = sim.save(e)
            assert probe.load(0, rec)
            probe.bt_rebuild(0)
            pcells, pspilled = probe.bt_owners(0)
            if not pspilled.any():
                continue
            assert (pcells == cells).all()
            assert probe.bt_count() & BT_SPILL
            assert all(probe.bt_flagged(0, int(c)) for c in cells)
            assert not any(probe.bt_flagged(0, int(c) ^ 1) for c in cells if int(c) ^ 1 not in set(cells.tolist()))
            h = sim.state_hash(e)
            assert sim.load(e, rec) and sim.state_hash(e) == h
            found = t
            break
    assert found is not None, "no arena overflowed the table at its rebuild"
