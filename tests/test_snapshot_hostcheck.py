"""Arena records (sf_save / sf_load) on the host-check build of the device code: the same layout table and
pack / unpack helpers (csrc/sf_snapshot.cuh) that the GPU kernels follow, so the GPU tests can compare
device records with these byte for byte.  The small capacities of test_split_step.py make many episodes
end, so a restored or cloned arena is followed across auto-resets; the tiny bullet-flag table variant
puts spill bits into the records."""
import numpy as np
import pytest

import common
import snapcheck
import sfo
from strikeforce_b200 import config as sfcfg
from test_split_step import CONFIGS, MAX_STEPS, N

BASE = 300
T1, T2 = 120, 260


def _actions(sim, t):
    return common.synth_actions(range(BASE, BASE + N), sim.n_agents, t, sfcfg.ACTIONS28).tobytes()


def _trace(sim, t0, steps):
    """step `steps` times from global step t0; per step: hash, step_out and status of every arena"""
    out = []
    for t in range(t0, t0 + steps):
        sim.step(_actions(sim, t))
        out.append([(sim.state_hash(e), tuple(sim.step_out(e).values()), sim.status(e)) for e in range(N)])
    return out


@pytest.mark.parametrize("name", list(CONFIGS))
def test_restore_in_place_and_resume(arena_data, name):
    """Step T1, save every arena, step T2, load the records back, replay T2 with the same actions: every step
    of every arena equals the first run, across auto-resets.  A fresh simulator of the same configuration that
    loads the T1 records follows the same trajectory (checkpoint and resume), and saving a loaded arena gives
    the loaded bytes back."""
    kw, extra = CONFIGS[name]
    cfg = sfcfg.make_config(arena_data, n_envs=N, auto_reset=True, max_steps=MAX_STEPS, env_id_base=BASE, **kw)
    a = snapcheck.SnapSim(cfg, extra=extra)
    _trace(a, 0, T1)
    recs = [a.save(e) for e in range(N)]
    first = _trace(a, T1, T2)
    ends = sum(so[0] != sfcfg.RUNNING for step in first for (_, so, _) in step)
    assert ends >= 10, "only %d episodes ended after the save" % ends
    for e in range(N):
        assert a.load(e, recs[e])
        assert (a.save(e) == recs[e]).all(), "save after load: arena %d" % e
    b = snapcheck.SnapSim(cfg, extra=extra)
    for e in range(N):
        assert b.load(e, recs[e])
    assert _trace(a, T1, T2) == first
    assert _trace(b, T1, T2) == first
    assert b.stats()["steps"] + b.stats()["overflows"] + b.stats()["ub_guards"] == N * T2, "b counts only its own steps"


def _oracle(arena_data, kw, level):
    return sfo.Arena(sfcfg.make_config(arena_data, mode=kw["mode"], level_min=level, squad_agents=kw.get("squad_agents", False),
                                       caps=kw["caps"], max_steps=MAX_STEPS, player=kw.get("player", "account1")))


def _level(kw, ge):
    lo = kw.get("level_min", 1)
    return lo + ge % (kw.get("level_max", lo) - lo + 1)


@pytest.mark.parametrize("name", ["solo", "timer", "squad-agents"])
def test_clone_follows_the_oracle(arena_data, name):
    """Arena 3 is followed by the C oracle from its first step.  At T1 it is cloned into arena 11 (another
    global id); the oracle then follows arena 11: the current episode goes on bit for bit, and at every episode
    end the oracle is reset with arena 11's level and seeds synth(ge_dst, episode + 1), the episode counter
    carried over from the source."""
    kw, extra = CONFIGS[name]
    src, dst = 3, 11
    cfg = sfcfg.make_config(arena_data, n_envs=N, auto_reset=True, max_steps=MAX_STEPS, env_id_base=BASE, **kw)
    sim = snapcheck.SnapSim(cfg, extra=extra)
    o = _oracle(arena_data, kw, _level(kw, BASE + src))
    ge, episode = BASE + src, 0
    o.reset(_level(kw, ge), common.synth_tb(ge), common.synth_serial(ge, 0))
    dst_ends = 0
    for t in range(T1 + 600):
        if t == T1:
            assert sim.load(dst, sim.save(src))
            ge = BASE + dst
            assert sim.state_hash(dst) == sim.state_hash(src)
        act = common.synth_actions(range(BASE, BASE + N), sim.n_agents, t, sfcfg.ACTIONS28)
        e = src if t < T1 else dst
        sim.step(act.tobytes())
        st = o.step(bytes(act[e]))
        assert sim.step_out(e)["status"] == st, "status: step %d" % t
        if st != sfcfg.RUNNING:
            episode += 1
            dst_ends += t >= T1
            o.reset(_level(kw, ge), common.synth_tb(ge), common.synth_serial(ge, episode))
        assert np.uint64(sim.state_hash(e)) == np.uint64(o.state_hash()), "state: step %d arena %d" % (t, e)
    assert dst_ends >= 3, "only %d episodes of the clone ended" % dst_ends


def test_incompatible_records_are_refused(arena_data):
    """A record is refused (and the arena left as it was) when it comes from other capacities, another mode or
    another Battle Royale ind.  n_envs, env_id_base, auto_reset, max_steps and the level range are not part of
    the fingerprint: such a record loads."""
    kw, _ = CONFIGS["squad-agents"]
    base = sfcfg.make_config(arena_data, n_envs=N, auto_reset=True, max_steps=MAX_STEPS, env_id_base=BASE, **kw)
    sim = snapcheck.SnapSim(base)
    sim.step(_actions(sim, 0))
    before = [sim.state_hash(e) for e in range(N)]
    caps = dict(kw["caps"], cap_zombies=kw["caps"]["cap_zombies"] + 1)
    royale = dict(mode=sfcfg.MODE_ROYALE, teams=[1, 2, 3, 4], caps=kw["caps"])
    others = {
        "caps": dict(kw, caps=caps),
        "cap_chests": dict(kw, caps=dict(kw["caps"], cap_chests=77)),  # not in the layout, same record size
        "mode": dict(kw, mode=sfcfg.MODE_SOLO, squad_agents=False),
        "squad_agents": dict(kw, squad_agents=False),
    }
    for what, okw in others.items():
        other = snapcheck.SnapSim(sfcfg.make_config(arena_data, n_envs=N, env_id_base=BASE, **okw))
        rec = np.resize(other.save(0), sim.snapshot_bytes)  # the header is checked first, whatever the size
        assert not sim.load(0, rec), what
    r0 = snapcheck.SnapSim(sfcfg.make_config(arena_data, n_envs=2, ind=0, **royale))
    r1 = snapcheck.SnapSim(sfcfg.make_config(arena_data, n_envs=2, ind=1, **royale))
    assert r0.snapshot_bytes == r1.snapshot_bytes
    assert not r0.load(0, r1.save(0)) and r0.load(0, r0.save(1))
    bad = sim.save(0)
    bad[0] ^= 1  # magic
    assert not sim.load(1, bad)
    assert [sim.state_hash(e) for e in range(N)] == before
    same = snapcheck.SnapSim(sfcfg.make_config(arena_data, n_envs=N + 40, auto_reset=False, max_steps=0, env_id_base=7,
                                               **dict(kw, level_min=3, level_max=4)))
    assert same.snapshot_bytes == sim.snapshot_bytes
    assert same.load(5, sim.save(2)) and same.state_hash(5) == sim.state_hash(2)
