"""Per-agent step outputs (sf_enable_agent_out, DESIGN.md section 7g) on the host-check build of the device tick.

The configurations, seeds and small capacities are those of test_split_step.py (Solo, Timer, Squad with agents with
the default and a tiny flag table, 16-player Battle Royale), so that many episodes end, some in an abort.  The
actions are the synthetic 28-symbol stream with '_' added, so that driven humans also quit.  Every test runs the
whole step, the split step and the list step (a permutation of all arenas with repeated and out-of-range ids).

- The rows equal rows built from an independent source: the canonical records (SF_K_HUMAN Hp, kills, damage,
  effect and active) and the action masks taken before and after every step.
- With auto-reset the rows equal those of the twin without auto-reset that resets its finished arenas after
  every step, and row ind equals sf_step_out wherever it is DRIVEN.
- Agent outputs change nothing else: sf_step_out, state hashes, statistics and records.
- A list step leaves the rows of unlisted arenas alone; S then its complement equals one whole step.
- The header's constants equal the Python mirror."""
import os
import re

import numpy as np
import pytest

import agentcheck
import common
from strikeforce_b200 import config as sfcfg
from test_split_step import BASE, CONFIGS, MAX_STEPS, N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEPS = 300
MAX_STEPS_HERE = 40  # well below test_split_step's 150: every arena ends several episodes
TABLE = sfcfg.ACTIONS28 + b"_"
ABORTS = (sfcfg.OVERFLOW, sfcfg.UB_GUARD)
PATHS = ("step", "split", "list")
# SF_K_HUMAN fields (include/sf_canon.h): active .. Hp(7) mindamage stamina kills(10) damage(11) effect(12)
H_ACTIVE, H_HP, H_KILLS, H_DMG, H_EFF = 0, 7, 10, 11, 12
DRIVEN, DIED = sfcfg.AGENT_DRIVEN, sfcfg.AGENT_DIED


def _sim(arena_data, name, auto_reset, agent_out=True):
    kw, extra = CONFIGS[name]
    cfg = sfcfg.make_config(arena_data, n_envs=N, auto_reset=auto_reset, max_steps=MAX_STEPS_HERE, env_id_base=BASE, **kw)
    return agentcheck.AgentSim(cfg, extra=agentcheck.EXTRA + tuple(extra), agent_out=agent_out)


def _actions(n_agents, t):
    return common.synth_actions(range(BASE, BASE + N), n_agents, t, TABLE)


def _list(rng):
    """all arenas in a random order, then repeated ids (with '_' rows) and out-of-range ids"""
    ids = rng.permutation(N)
    extra = np.concatenate([rng.choice(N, size=rng.integers(0, 4)), np.array([-1, N])[:rng.integers(0, 3)]])
    return np.concatenate([ids, extra]).astype(np.int32), len(ids)


def _step(sim, act, path, rng):
    """one step of every arena through `path`"""
    if path == "step":
        sim.step(act.tobytes())
    elif path == "split":
        sim.step(None, half=1)
        sim.step(act.tobytes(), half=2)
    else:
        ids, n_live = _list(rng)
        rows = np.full((len(ids), sim.n_agents), ord("_"), np.uint8)
        rows[:n_live] = act[ids[:n_live]]
        sim.step_list(rows, ids)


def _humans(sim, env):
    """{slot: SF_K_HUMAN fields} of the arena's canonical record"""
    rec, out, i = sim.dump(env), {}, 0
    while i + 3 <= len(rec):
        kind, index, nf = int(rec[i]), int(rec[i + 1]), int(rec[i + 2])
        if kind == 3:
            out[index] = rec[i + 3:i + 3 + nf].copy()
        i += 3 + nf
    return out


def _expected(sim, before, masks):
    """the rows of the last step from the records before (`before`, per arena), the masks before (`masks`) and the
    records now"""
    want = np.zeros((N, sim.n_agents, 5), np.int32)
    for e in range(N):
        after = _humans(sim, e)
        for a in range(sim.n_agents):
            if masks[e, a] == 0:
                continue
            h0, h1 = before[e][a], after[a]  # a driven slot is live at the start, so in both records
            want[e, a] = (DRIVEN | (0 if h1[H_ACTIVE] else DIED), h1[H_HP] - h0[H_HP], h1[H_DMG] - h0[H_DMG],
                          h1[H_EFF] - h0[H_EFF], h1[H_KILLS] - h0[H_KILLS])
    return want


def _compare(got, want, aborted, what):
    for e in range(N):
        if aborted[e]:  # only DRIVEN is defined
            ok = ((got[e, :, 0] & DRIVEN) == (want[e, :, 0] & DRIVEN)).all()
        else:
            ok = (got[e] == want[e]).all()
        assert ok, "%s arena %d: %s vs %s" % (what, e, got[e].tolist(), want[e].tolist())


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", list(CONFIGS))
def test_rows_equal_the_definition_from_records(arena_data, name, path):
    """auto_reset = 0 and hc_reset_finished after every step, so that the record at the end of a step can be read.
    The expected rows come from the records and the masks alone: DRIVEN = mask word != 0 before the step, d_* from
    the SF_K_HUMAN fields, DIED from `active` after the step.  Row ind also equals sf_step_out where DRIVEN."""
    sim = _sim(arena_data, name, auto_reset=False)
    rng = np.random.default_rng(sum(map(ord, name + path)))
    ind = CONFIGS[name][0].get("ind", 0)
    seen = dict(driven=0, died=0, ended=0, aborted=0, idle=0)
    for t in range(STEPS):
        act = _actions(sim.n_agents, t)
        masks = sim.masks()
        before = [_humans(sim, e) for e in range(N)]
        _step(sim, act, path, rng)
        got = sim.agent_out()
        status = np.array([sim.status(e) for e in range(N)])
        aborted = np.isin(status, ABORTS)
        _compare(got, _expected(sim, before, masks), aborted, "%s %s step %d" % (name, path, t))
        for e in range(N):
            o = sim.step_out(e)
            if got[e, ind, 0] & DRIVEN and not aborted[e]:
                assert (o["d_hp"], o["d_damage"], o["d_effect"]) == tuple(got[e, ind, 1:4]), "step_out, arena %d" % e
        seen["driven"] += int((got[:, :, 0] & DRIVEN != 0).sum())
        seen["died"] += int((got[:, :, 0] & DIED != 0).sum())
        seen["idle"] += int(((masks != 0) != (got[:, :, 0] != 0)).sum())  # must stay 0: DRIVEN is the mask
        seen["ended"] += int((status != sfcfg.RUNNING).sum())
        seen["aborted"] += int(aborted.sum())
        sim.reset_finished()
    assert seen["idle"] == 0
    assert seen["driven"] and seen["died"] and seen["ended"] >= N, seen


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", list(CONFIGS))
def test_auto_reset_rows_equal_reset_finished_twin(arena_data, name, path):
    """the rows of an auto_reset = 1 run equal those of its auto_reset = 0 twin that resets its finished arenas
    after every step, every step: DIED and the end values are read before the auto-reset"""
    auto, twin = _sim(arena_data, name, True), _sim(arena_data, name, False)
    r1, r2 = np.random.default_rng(7), np.random.default_rng(7)
    ind = CONFIGS[name][0].get("ind", 0)
    died = ended = 0
    for t in range(STEPS):
        act = _actions(auto.n_agents, t)
        _step(auto, act, path, r1)
        _step(twin, act, path, r2)
        got, want = auto.agent_out(), twin.agent_out()
        assert (got == want).all(), "%s %s step %d arena %d" % (name, path, t, np.nonzero((got != want).any((1, 2)))[0][0])
        for e in range(N):
            o = auto.step_out(e)
            ended += o["status"] != sfcfg.RUNNING
            if got[e, ind, 0] & DRIVEN and o["status"] not in ABORTS:
                assert (o["d_hp"], o["d_damage"], o["d_effect"]) == tuple(got[e, ind, 1:4])
        died += int((got[:, :, 0] & DIED != 0).sum())
        twin.reset_finished()
    assert died and ended >= N


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", list(CONFIGS))
def test_agent_out_changes_nothing_else(arena_data, name, path):
    """a handle with agent outputs and one without: sf_step_out and state hashes every step, the statistics, and
    the records at the end are equal"""
    on, off = _sim(arena_data, name, True), _sim(arena_data, name, True, agent_out=False)
    r1, r2 = np.random.default_rng(11), np.random.default_rng(11)
    for t in range(STEPS):
        act = _actions(on.n_agents, t)
        _step(on, act, path, r1)
        _step(off, act, path, r2)
        for e in range(N):
            assert on.state_hash(e) == off.state_hash(e), "%s %s step %d arena %d" % (name, path, t, e)
            assert on.step_out(e) == off.step_out(e)
    assert on.stats() == off.stats()
    for e in range(N):
        assert (on.save(e) == off.save(e)).all()


@pytest.mark.parametrize("name", list(CONFIGS))
def test_list_step_rows(arena_data, name):
    """stepping a subset S leaves the rows of every other arena as they were; S then its complement gives the rows
    of one whole step (reference: hc_step of all arenas)"""
    whole, parts = _sim(arena_data, name, True), _sim(arena_data, name, True)
    rng = np.random.default_rng(sum(map(ord, name)))
    for t in range(STEPS):
        act = _actions(whole.n_agents, t)
        whole.step(act.tobytes())
        inside = rng.random(N) < rng.random()
        for part in (np.nonzero(inside)[0], np.nonzero(~inside)[0]):
            prev = parts.agent_out()
            ids = np.concatenate([rng.permutation(part), [-1, N]]).astype(np.int32)
            rows = np.full((len(ids), whole.n_agents), ord("+"), np.uint8)
            rows[:len(part)] = act[ids[:len(part)]]
            parts.step_list(rows, ids)
            now = parts.agent_out()
            out = np.setdiff1d(np.arange(N), part)
            assert (now[out] == prev[out]).all(), "%s step %d: an unlisted arena's rows changed" % (name, t)
        got, want = parts.agent_out(), whole.agent_out()
        assert (got == want).all(), "%s step %d" % (name, t)


def test_header_mirrors_config():
    """SF_FIELD_AGENT_OUT, SF_AGENT_DRIVEN / SF_AGENT_DIED and the fields of sf_agent_out equal the Python mirror"""
    text = open(os.path.join(ROOT, "include", "strikeforce_b200.h")).read()
    assert int(re.search(r"SF_FIELD_AGENT_OUT\s*=\s*(\d+)", text).group(1)) == sfcfg.FIELD_AGENT_OUT
    assert int(re.search(r"SF_AGENT_DRIVEN\s*=\s*(\d+)", text).group(1)) == sfcfg.AGENT_DRIVEN
    assert int(re.search(r"SF_AGENT_DIED\s*=\s*(\d+)", text).group(1)) == sfcfg.AGENT_DIED
    body = re.search(r"typedef struct sf_agent_out \{(.*?)\} sf_agent_out;", text, re.S).group(1)
    assert tuple(re.findall(r"int32_t\s+(\w+);", body)) == sfcfg.AGENT_OUT_FIELDS
