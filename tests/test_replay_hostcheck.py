"""Replay (sf_enable_replay / sf_replay_load, DESIGN.md section 7i) on the host-check build of the device tick.

The configurations are those of test_match_log_hostcheck.py (Solo, Timer, Squad with agents with the default and a
tiny flag table, 16-player Battle Royale at ind = 5; episodes truncated at 40 steps).

- Round trip: complete tapes of episodes played on a logging handle, loaded into other arenas and into the same ones
  of a replay handle with logs on, replay every step's state hash with junk action rows, end with the recorded
  status, ENDED, cursor == n_symbols and no SURPLUS, and log the source row's head and symbols again (byte for byte
  in the same arena, all but global_id in another), through the whole, split and list steps.  The dealt rows are the tape split by
  the slots the C oracle logs between the halves.
- Short tapes follow the twin fed the first k symbols and then the rows; long tapes end in SURPLUS.
- Lists, refusals, duplicates and the disarming calls behave as defined; with no tape armed nothing changes; the
  header's constants equal the Python mirror; replay.tape_rows refuses logs the handle cannot replay."""
import os
import re

import numpy as np
import pytest

import logcheck
import replaycheck
import sfo
from strikeforce_b200 import config as sfcfg
from strikeforce_b200 import replay
from test_match_log_hostcheck import (ABORTS, CONFIGS, MAX_STEPS_HERE, _actions, _cfg, _delivered, needs_reference)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAP = 16 * MAX_STEPS_HERE
ARMED, EXHAUSTED, ENDED, SURPLUS = (sfcfg.REPLAY_ARMED, sfcfg.REPLAY_EXHAUSTED, sfcfg.REPLAY_ENDED,
                                    sfcfg.REPLAY_SURPLUS)
HEAD = sfcfg.LOG_HEAD.itemsize


def _sim(arena_data, name, auto_reset, n, replay=CAP, match_log=0, agent_out=False):
    return replaycheck.ReplaySim(_cfg(arena_data, name, auto_reset, n), extra=replaycheck.EXTRA + tuple(CONFIGS[name][1]),
                                 agent_out=agent_out, match_log=match_log, replay=replay)


def _record(arena_data, name, n=8, steps=160, seed=0):
    """episodes played with random rows on a logging handle (auto_reset = 0, sf_reset_finished): [(source arena,
    exported row, state hash after every step, final status)] of the complete, replayable ones"""
    sim = _sim(arena_data, name, False, n, replay=0, match_log=CAP)
    rng = np.random.default_rng(seed + len(name))
    hashes, out = [[] for _ in range(n)], []
    for _ in range(steps):
        running = [sim.status(e) == sfcfg.RUNNING for e in range(n)]
        sim.step(_actions(rng, n, sim.n_agents).tobytes())
        rows = sim.logs()
        for e in range(n):
            if not running[e]:
                continue
            hashes[e].append(sim.state_hash(e))
            if sim.status(e) != sfcfg.RUNNING:
                flags = int(logcheck.heads(rows[e:e + 1])[0]["flags"])
                if flags & sfcfg.LOG_COMPLETE and not flags & sfcfg.LOG_UNREPLAYABLE:
                    out.append((e, rows[e].copy(), hashes[e], sim.status(e)))
                hashes[e] = []
        sim.reset_finished()
    assert len(out) >= n
    return out


def _oracle_dealt(arena_data, name, row):
    """the tape split by the C oracle's logged set (the loop of _oracle_replay in test_match_log_hostcheck.py): for
    every step, {slot: symbol as delivered to obey}"""
    kw = CONFIGS[name][0]
    h = logcheck.heads(row[None])[0]
    royale = kw["mode"] == sfcfg.MODE_ROYALE
    if royale:
        ocfg = sfcfg.make_config(arena_data, mode=sfcfg.MODE_ROYALE, teams=kw["teams"], ind=kw["ind"], caps=kw["caps"],
                                 max_steps=MAX_STEPS_HERE)
    else:
        okw = {k: v for k, v in kw.items() if k not in ("level_min", "level_max")}
        ocfg = sfcfg.make_config(arena_data, level_min=int(h["level"]), max_steps=MAX_STEPS_HERE, **okw)
    o = sfo.Arena(ocfg)
    o.reset(int(h["level"]), int(h["tb"]), int(h["serial"]))
    tape = logcheck.tape(row)
    n_agents = 16 if royale else (10 if kw.get("squad_agents") else 1)
    ind = kw.get("ind", 0)
    pos, out = 0, []
    while pos < len(tape):
        dealt = {}
        if o.step_a() == sfcfg.RUNNING:
            rec = sfo.parse_record(o.dump())
            logged = [ind] + [a for a in range(n_agents) if a != ind and (3, a) in rec and rec[(3, a)][0]
                              and not rec[(3, a)][1]]
            row_a = bytearray(b"+" * n_agents)
            for a in logged:
                row_a[a] = tape[pos]
                dealt[a] = tape[pos] if a == ind else _delivered(name, a, tape[pos])
                pos += 1
            o.step_b(bytes(row_a))
        out.append(dealt)
    return out


def _step(sim, act, path, n):
    if path == "step":
        sim.step(act.tobytes())
    elif path == "split":
        sim.step(None, half=1)
        sim.step(act.tobytes(), half=2)
    else:  # a list in reverse order with a repeat and ids out of range: the same step for every arena
        ids = np.concatenate([np.arange(n)[::-1], [0, -1, n]]).astype(np.int32)
        rows = np.full((len(ids), sim.n_agents), ord("_"), np.uint8)
        rows[:n] = act[ids[:n]]
        sim.step_list(rows, ids)


@pytest.mark.parametrize("path", ["step", "split", "list"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_round_trip(arena_data, name, path):
    n = 8
    episodes = _record(arena_data, name, n)
    sim = _sim(arena_data, name, False, n, match_log=CAP)
    rng = np.random.default_rng(99)
    checked_dealt = 0
    for r in range(0, min(len(episodes), 3 * n), n):
        batch = episodes[r:r + n]
        # the first round loads every tape back into its own arena where it can, later rounds shift them
        targets = [(src + r // n) % n for src, _, _, _ in batch]
        seen = set()
        for i, t in enumerate(targets):
            while t in seen:
                t = (t + 1) % n
            targets[i] = t
            seen.add(t)
        rows = np.stack([row for _, row, _, _ in batch])
        assert sim.replay_load(rows, targets) == 0
        dealt_want = {t: _oracle_dealt(arena_data, name, row) for t, (_, row, _, _) in zip(targets, batch)} \
            if path == "step" else {}
        for step in range(max(len(h) for _, _, h, _ in batch)):
            _step(sim, _actions(rng, n, sim.n_agents), path, n)
            for t, (src, row, hashes, status) in zip(targets, batch):
                if step < len(hashes):
                    assert sim.state_hash(t) == hashes[step], "%s %s: arena %d left the episode at step %d" % (
                        name, path, t, step)
                if t in dealt_want and step < len(dealt_want[t]):
                    want = np.zeros(sim.n_agents, np.uint8)
                    for a, c in dealt_want[t][step].items():
                        want[a] = c
                    assert (sim.replay_dealt(t) == want).all(), "%s arena %d step %d" % (name, t, step)
                    checked_dealt += 1
        logs = sim.logs()
        for t, (src, row, hashes, status) in zip(targets, batch):
            h = logcheck.heads(row[None])[0]
            assert sim.replay_state(t) == (ENDED, int(h["n_symbols"]), int(h["n_symbols"]), len(hashes) -
                                           (status in ABORTS), status), (name, path, t)
            assert sim.status(t) == status
            got = logs[t].copy()
            if t != src:
                got[HEAD - 8:HEAD] = row[HEAD - 8:HEAD]  # global_id, the last field of the head
                assert int(logcheck.heads(logs[t:t + 1])[0]["global_id"]) != int(h["global_id"])
            n_sym = HEAD + int(h["n_symbols"])  # the head and the symbols: what is past them is a tape's old content
            assert (got[:n_sym] == row[:n_sym]).all(), "%s %s: the log of arena %d differs from the source row" % (
                name, path, t)
        sim.reset_finished()
    assert path != "step" or checked_dealt


def _twin_expected(ref, act, tape, pos, ind, name):
    """step a replay-less twin half by half, the first tape symbols going to the logged slots (ind, then the slots
    whose action mask is not 0 at P2); returns the new position in the tape"""
    ref.step(None, half=1)
    masks = ref.masks()
    row = act.copy()
    if ref.status(0) == sfcfg.RUNNING:
        for a in [ind] + [a for a in range(ref.n_agents) if a != ind and masks[0, a] != 0]:
            if pos >= len(tape):
                break
            row[0, a] = tape[pos]
            pos += 1
    ref.step(row.tobytes(), half=2)
    return pos


@pytest.mark.parametrize("name", list(CONFIGS))
def test_short_and_long_tapes(arena_data, name):
    src, row, hashes, status = _record(arena_data, name, 4, seed=5)[0]
    n_sym = int(logcheck.heads(row[None])[0]["n_symbols"])
    ind = CONFIGS[name][0].get("ind", 0)
    rng = np.random.default_rng(17)
    for k in (0, 1, n_sym // 2):
        cut = row.copy()
        cut[HEAD + k:] = 0
        cut[HEAD - 28:HEAD - 24] = np.frombuffer(np.int32(k).tobytes(), np.uint8)  # n_symbols
        assert int(logcheck.heads(cut[None])[0]["n_symbols"]) == k
        sim, ref = _sim(arena_data, name, False, 1), _sim(arena_data, name, False, 1)
        assert sim.replay_load(cut[None], [0]) == 0
        # the twin starts from the same load with an empty tape: it deals nothing and plays the rows it is given
        empty = cut.copy()
        empty[HEAD - 28:HEAD - 24] = 0
        assert ref.replay_load(empty[None], [0]) == 0 and ref.state_hash(0) == sim.state_hash(0)
        tape, pos, exhausted_at = logcheck.tape(row)[:k], 0, None
        for t in range(MAX_STEPS_HERE):
            if sim.status(0) != sfcfg.RUNNING:
                break
            act = _actions(rng, 1, sim.n_agents)
            before = pos
            pos = _twin_expected(ref, act, tape, pos, ind, name)
            sim.step(act.tobytes())
            assert sim.state_hash(0) == ref.state_hash(0), "%s k=%d step %d" % (name, k, t)
            flags = sim.replay_state(0)[0]
            if exhausted_at is None and (flags & EXHAUSTED):
                exhausted_at = t
                assert not flags & ARMED and pos == k and before <= k
            elif exhausted_at is None:
                assert flags & ARMED or flags & ENDED
        assert exhausted_at is not None or sim.replay_state(0)[0] & ENDED
    # appended symbols: the episode ends with symbols left over
    long = row.copy()
    long[HEAD + n_sym:HEAD + n_sym + 3] = np.frombuffer(b"+++", np.uint8)
    long[HEAD - 28:HEAD - 24] = np.frombuffer(np.int32(n_sym + 3).tobytes(), np.uint8)
    sim = _sim(arena_data, name, False, 1)
    assert sim.replay_load(long[None], [0]) == 0
    for _ in range(len(hashes)):
        sim.step(_actions(rng, 1, sim.n_agents).tobytes())
    assert sim.replay_state(0) == (ENDED | SURPLUS, n_sym, n_sym + 3, len(hashes) - (status in ABORTS), status)


def _rows(arena_data, name, n, seed=1):
    return np.stack([row for _, row, _, _ in _record(arena_data, name, 8, seed=seed)[:n]])


def test_list_step_leaves_unlisted_tapes_alone(arena_data):
    name, n = "squad-agents", 8
    rows = _rows(arena_data, name, n)
    sim = _sim(arena_data, name, False, n)
    assert sim.replay_load(rows, np.arange(n)) == 0
    rng = np.random.default_rng(3)
    for t in range(10):
        part = np.nonzero(rng.random(n) < 0.5)[0]
        before = [sim.replay_state(e) for e in range(n)]
        dealt = [sim.replay_dealt(e).copy() for e in range(n)]
        hashes = [sim.state_hash(e) for e in range(n)]
        sim.step_list(_actions(rng, len(part), sim.n_agents), part)
        for e in np.setdiff1d(np.arange(n), part):
            assert sim.replay_state(e) == before[e] and (sim.replay_dealt(e) == dealt[e]).all()
            assert sim.state_hash(e) == hashes[e]
        for e in part:
            if before[e][0] & ARMED:
                assert sim.replay_state(e)[1] > before[e][1], "a listed armed arena dealt nothing"


def test_refusals_are_all_or_nothing_and_duplicates_load_once(arena_data):
    name, n = "solo", 4
    rows = _rows(arena_data, name, n)
    sim = _sim(arena_data, name, False, n)
    hashes = [sim.state_hash(e) for e in range(n)]

    def with_head(row, **kw):
        r = row.copy()
        h = r[:HEAD].view(sfcfg.LOG_HEAD)
        for k, v in kw.items():
            h[k] = v
        return r

    bad = [with_head(rows[0], level=0), with_head(rows[1], level=65),  # SF_MAX_LEVEL = 64
           with_head(rows[2], tb=-1), with_head(rows[3], serial=-5), with_head(rows[0], n_symbols=CAP + 1),
           with_head(rows[1], n_symbols=-1)]
    for b in bad:
        assert sim.replay_load(np.stack([rows[2], b]), [2, 1]) == 1
        assert [sim.state_hash(e) for e in range(n)] == hashes and all(sim.replay_state(e)[0] == 0 for e in range(n))
    assert sim.replay_load(np.stack(bad[:3]), [0, 1, 2]) == 3
    # a refused entry that does not own its id, and ids out of range, do not count
    assert sim.replay_load(np.stack([rows[0], bad[0], rows[1], rows[2]]), [3, 3, -1, n]) == 0
    assert sim.replay_state(3)[0] == ARMED and sim.replay_state(3)[2] == int(logcheck.heads(rows[:1])[0]["n_symbols"])
    assert [sim.replay_state(e)[0] for e in range(3)] == [0, 0, 0]
    # royale plays level 1 only
    rsim = _sim(arena_data, "royale16", False, 2)
    rrows = _rows(arena_data, "royale16", 2)
    assert rsim.replay_load(np.stack([rrows[0], with_head(rrows[1], level=2)]), [0, 1]) == 1
    assert rsim.replay_load(rrows, [0, 1]) == 0


def test_reset_and_loads_disarm(arena_data):
    name, n = "squad-agents", 4
    rows = _rows(arena_data, name, n)
    sim = _sim(arena_data, name, False, n)
    armed = lambda: [sim.replay_state(e)[0] & ARMED for e in range(n)]  # noqa: E731
    assert sim.replay_load(rows, np.arange(n)) == 0 and armed() == [ARMED] * n
    sim.reset(1, 5, 6)
    assert armed() == [ARMED, 0, ARMED, ARMED]
    rec = sim.save(3)
    assert sim.load(2, rec) and armed() == [ARMED, 0, 0, ARMED]
    bad = rec.copy()
    bad[:4] ^= 0xFF
    assert sim.load_list(np.stack([rec, bad]), [0, 3], rows=[0, 1]) == 1 and armed() == [ARMED, 0, 0, ARMED]
    assert sim.load_list(np.stack([rec]), [3], rows=[0]) == 0 and armed() == [ARMED, 0, 0, 0]
    sim.reset_finished()  # touches no replay state
    assert armed() == [ARMED, 0, 0, 0]


@pytest.mark.parametrize("path", ["step", "split"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_replay_without_a_tape_changes_nothing(arena_data, name, path):
    """a replay handle with logs and agent outputs on against the same handle without replay, 300 steps with
    auto-reset: state hashes, sf_step_out, agent rows, logs, statistics and records"""
    n = 8
    on = _sim(arena_data, name, True, n, match_log=CAP, agent_out=True)
    off = _sim(arena_data, name, True, n, replay=0, match_log=CAP, agent_out=True)
    rng = np.random.default_rng(31)
    for t in range(300):
        act = _actions(rng, n, on.n_agents)
        for s in (on, off):
            _step(s, act, path, n)
        assert (on.agent_out() == off.agent_out()).all(), "%s %s step %d" % (name, path, t)
        for e in range(n):
            assert on.state_hash(e) == off.state_hash(e) and on.step_out(e) == off.step_out(e), (name, path, t)
            assert not on.replay_dealt(e).any() and on.replay_state(e) == (0, 0, 0, 0, 0)
    assert (on.logs() == off.logs()).all() and on.stats() == off.stats()
    for e in range(n):
        assert (on.save(e) == off.save(e)).all()


def test_enable_replay_arguments(arena_data):
    sim = _sim(arena_data, "solo", False, 2, replay=0)
    assert sim.replay_row_bytes == 0
    assert not sim.enable_replay(0) and not sim.enable_replay(sfcfg.LOG_CAP_MAX + 1)
    assert sim.enable_replay(100) and sim.enable_replay(100) and not sim.enable_replay(101)
    assert sim.replay_row_bytes == sfcfg.replay_row_bytes(100) == sfcfg.log_row_bytes(100)


def test_header_mirrors_config():
    """SF_REPLAY_*, the SF_FIELD_REPLAY* numbers and the fields of sf_replay_state equal the Python mirror"""
    text = open(os.path.join(ROOT, "include", "strikeforce_b200.h")).read()
    for name in ("ARMED", "EXHAUSTED", "ENDED", "SURPLUS"):
        assert int(re.search(r"SF_REPLAY_%s\s*=\s*(\d+)" % name, text).group(1)) == getattr(sfcfg, "REPLAY_" + name)
    assert int(re.search(r"SF_FIELD_REPLAY\s*=\s*(\d+)", text).group(1)) == sfcfg.FIELD_REPLAY
    assert int(re.search(r"SF_FIELD_REPLAY_DEALT\s*=\s*(\d+)", text).group(1)) == sfcfg.FIELD_REPLAY_DEALT
    body = re.search(r"typedef struct sf_replay_state \{(.*?)\} sf_replay_state;", text, re.S).group(1)
    assert tuple(re.findall(r"int32_t\s+(\w+);", body)) == sfcfg.REPLAY_STATE.names
    assert all(sfcfg.REPLAY_STATE[f] == np.dtype("<i4") for f in sfcfg.REPLAY_STATE.names)


def test_tape_rows_from_files(arena_data, tmp_path):
    """a device row written as a file and read back gives the same load row (global id and flags aside), and
    tape_rows refuses what the handle cannot replay"""
    for name in ("solo", "squad-agents", "royale16"):
        cfg = _cfg(arena_data, name, False, 1)
        _, row, _, _ = _record(arena_data, name, 4, seed=2)[0]
        path = str(tmp_path / ("%s.sf_sample" % name))
        level = replay.write_device_log(path, row, cfg)
        log = replay.read_royale(path) if name == "royale16" else replay.read(path)
        got = replay.tape_rows([log], cfg, CAP, level)[0]
        want = row.copy()
        want[:HEAD].view(sfcfg.LOG_HEAD)[["flags", "status", "steps", "global_id", "episode"]] = 0
        assert (got == want).all(), name
        with pytest.raises(ValueError):
            replay.tape_rows([log], cfg, len(log.commands) - 1, level)
        if name == "royale16":
            with pytest.raises(ValueError):
                replay.tape_rows([log], _cfg(arena_data, "solo", False, 1), CAP)
            other = replay.RoyaleLog(log.server, log.tb, log.serial, 4, log.teams, log.names, log.sheets, log.commands)
            with pytest.raises(ValueError):
                replay.tape_rows([other], cfg, CAP)
            other = replay.RoyaleLog(log.server, log.tb, log.serial, log.ind, log.teams[::-1], log.names, log.sheets,
                                     log.commands)
            with pytest.raises(ValueError):
                replay.tape_rows([other], cfg, CAP)
        else:
            with pytest.raises(ValueError):
                replay.tape_rows([log], _cfg(arena_data, "royale16", False, 1), CAP)
            sheet = log.sheet.copy()
            sheet[0] += 1
            with pytest.raises(ValueError):
                replay.tape_rows([replay.MatchLog(log.tb, log.serial, 1, 0, 1, log.name, sheet, log.commands)], cfg, CAP)
            with pytest.raises(ValueError):
                replay.tape_rows([replay.MatchLog(log.tb, log.serial, 2, 0, 1, log.name, log.sheet, log.commands)], cfg,
                                 CAP)


@needs_reference
def test_a_reference_written_file_replays_to_the_reference_record(arena_data, tmp_path):
    """a file written by the reference's own logger, read with replay.read and loaded through tape_rows, ends in
    the reference's final record (default caps, so that nothing overflows)"""
    import sfref
    level, steps = 2, 120
    cfg = sfcfg.make_config(arena_data, n_envs=1, mode=sfcfg.MODE_SQUAD, level_min=level, squad_agents=True,
                            auto_reset=False)
    caps = [sfcfg.DEFAULT_CAPS[k] for k in ("cap_humans", "cap_zombies", "cap_bullets", "cap_chests", "cap_built",
                                            "cap_portals")]
    sfref.reset_logging(sfcfg.MODE_SQUAD, level, squad_agents=True, caps=caps)
    rng = np.random.default_rng(8)
    for _ in range(steps):
        if sfref.step(np.frombuffer(sfcfg.ACTIONS9, np.uint8)[rng.integers(9, size=10)].tobytes()) != 0:
            break
    want = sfref.dump()
    path = sfref.close_log()
    log = replay.read(path)
    os.remove(path)
    sim = replaycheck.ReplaySim(cfg, replay=len(log.commands) + 16)
    assert sim.replay_load(replay.tape_rows([log], cfg, len(log.commands) + 16, level), [0]) == 0
    junk = np.frombuffer(b"_", np.uint8)
    while sim.replay_state(0)[0] & ARMED and sim.replay_state(0)[1] < len(log.commands):  # not a step past the tape
        sim.step(np.repeat(junk, sim.n_agents).tobytes())
    got = sim.dump(0)
    assert len(got) == len(want) and (got == want).all()


GOLDEN = ["squad_l3_agents", "royale_5p_ind2", "royale_4p_ind3_short", "royale_16p_4teams"]


@pytest.mark.parametrize("golden", GOLDEN)
def test_tapes_of_reference_trajectories_reach_the_golden_hashes(arena_data, golden):
    """the golden match's actions, split into a tape by the C oracle's logged set between the halves, loaded into
    arena 1 and played with junk rows, reach the reference's hash after every step"""
    import common
    g = np.load(os.path.join(ROOT, "tests", "golden", golden + ".npz"))
    kw = common.golden_kwargs(g)
    level, tb, serial = int(g["level"]), int(g["tb"]), int(g["serial"])
    o = sfo.Arena(sfcfg.make_config(arena_data, level_min=level, **kw))
    o.reset(level, tb, serial)
    n_agents, ind = g["actions"].shape[1], int(g["ind"]) if "ind" in g else 0
    royale = kw["mode"] == sfcfg.MODE_ROYALE
    tape = bytearray()
    for act in g["actions"]:
        if o.step_a() == sfcfg.RUNNING:
            rec = sfo.parse_record(o.dump())
            tape.append(int(act[ind]))
            for a in range(n_agents):
                if a != ind and (3, a) in rec and rec[(3, a)][0] and not rec[(3, a)][1]:
                    c = int(act[a])
                    tape.append(c if royale or c in sfcfg.ACTIONS9 else ord("+"))
        o.step_b(bytes(act))
    cap = len(tape) + 16
    row = np.zeros(sfcfg.replay_row_bytes(cap), np.uint8)
    head = row[:HEAD].view(sfcfg.LOG_HEAD)
    head["level"], head["n_symbols"], head["tb"], head["serial"] = level, len(tape), tb, serial
    row[HEAD:HEAD + len(tape)] = np.frombuffer(bytes(tape), np.uint8)
    sim = replaycheck.ReplaySim(sfcfg.make_config(arena_data, n_envs=2, level_min=level, auto_reset=False, **kw),
                                replay=cap)
    assert sim.replay_load(row[None], [1]) == 0
    assert np.uint64(sim.state_hash(1)) == g["hashes"][0]
    junk = np.frombuffer(b"_3u", np.uint8)
    rng = np.random.default_rng(0)
    for t in range(len(g["actions"])):
        sim.step(junk[rng.integers(3, size=2 * sim.n_agents)].tobytes())
        assert sim.status(1) == g["status"][t], "%s status, step %d" % (golden, t)
        assert np.uint64(sim.state_hash(1)) == g["hashes"][t + 1], "%s state hash, step %d" % (golden, t)
    state = sim.replay_state(1)
    assert state[1] == len(tape) and not state[0] & SURPLUS
