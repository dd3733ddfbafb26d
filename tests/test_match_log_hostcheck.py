"""Match logs (sf_enable_log / sf_log_list, DESIGN.md section 7h) on the host-check build of the device tick.

The configurations and small capacities are those of test_split_step.py (Solo, Timer, Squad with agents with the
default and a tiny flag table) with the 16-player Battle Royale at ind = 5, episodes truncated at 40 steps, and
random action rows over all 30 symbols, so that squad agents are given symbols that reach obey as '+'.

- The tapes equal the stream built independently between the halves of a twin: ind's symbol, then every slot whose
  action mask is not 0 at P2 with its delivered symbol -- the construction the reference-logger test of
  test_replay_format.py uses -- with the episode's seeds, level, episode counter, step count and final status.
- Every complete tape, written as a .sf_sample file and read back, is replayed by the C oracle from the header's
  seeds and level to the recorded arena's state hash after every step and to its final status; where the
  reference is built, its own reader replays a Solo and a Squad-with-agents file to the same final record.
- Seeds round-trip; the flags (load, truncation, aborts, junk bytes) and the list step behave as defined; logs
  change nothing else; the header's constants equal the Python mirror."""
import os
import re

import numpy as np
import pytest

import common
import logcheck
import sfo
import sfref
from strikeforce_b200 import config as sfcfg
from strikeforce_b200 import replay
from test_split_step import BASE, N, ROYALE_CAPS, SMALL, SPILL_STRESS, SQUAD_CAPS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEPS = 300
MAX_STEPS_HERE = 40
CAP = 16 * MAX_STEPS_HERE  # never full: at most 16 symbols a step
CONFIGS = {
    "solo": (dict(mode=sfcfg.MODE_SOLO, level_min=1, level_max=10, caps=SMALL), ()),
    "timer": (dict(mode=sfcfg.MODE_TIMER, level_min=1, level_max=10, caps=SMALL, player="synthetic"), ()),
    "squad-agents": (dict(mode=sfcfg.MODE_SQUAD, level_min=1, level_max=10, squad_agents=True, caps=SQUAD_CAPS), ()),
    "squad-agents-tiny-flag-table": (dict(mode=sfcfg.MODE_SQUAD, level_min=1, level_max=10, squad_agents=True,
                                          caps=SQUAD_CAPS), SPILL_STRESS),
    "royale16": (dict(mode=sfcfg.MODE_ROYALE, teams=[1, 2, 3, 4] * 4, caps=ROYALE_CAPS, ind=5), ()),
}
ABORTS = (sfcfg.OVERFLOW, sfcfg.UB_GUARD)
JUNK = b"\x00 \t\n\x0b\x0c\r"
COMPLETE, TRUNCATED, ABORTED, UNREPLAYABLE = (sfcfg.LOG_COMPLETE, sfcfg.LOG_TRUNCATED, sfcfg.LOG_ABORTED,
                                              sfcfg.LOG_UNREPLAYABLE)
needs_reference = pytest.mark.skipif(not sfref.available(), reason="oracle/_ref/libsfref.so not built")


def _cfg(arena_data, name, auto_reset, n=N, **over):
    kw = dict(CONFIGS[name][0], **over)
    return sfcfg.make_config(arena_data, n_envs=n, auto_reset=auto_reset, max_steps=MAX_STEPS_HERE, env_id_base=BASE,
                             **kw)


def _sim(arena_data, name, auto_reset, match_log=CAP, agent_out=False, n=N):
    return logcheck.LogSim(_cfg(arena_data, name, auto_reset, n), extra=logcheck.EXTRA + tuple(CONFIGS[name][1]),
                           agent_out=agent_out, match_log=match_log)


def _actions(rng, n, n_agents):
    return np.frombuffer(sfcfg.COMMANDS, np.uint8)[rng.integers(len(sfcfg.COMMANDS), size=(n, n_agents))]


def _level(name, e):
    kw = CONFIGS[name][0]
    if kw["mode"] == sfcfg.MODE_ROYALE:
        return 1
    lo = kw.get("level_min", 1)
    return lo + (BASE + e) % (kw.get("level_max", lo) - lo + 1)


def _delivered(name, a, c):
    """what obey receives for a logged slot a != ind: a squad agent's symbol outside "+xzqeawsd" arrives as '+'"""
    if CONFIGS[name][0]["mode"] != sfcfg.MODE_ROYALE and c not in sfcfg.ACTIONS9:
        return ord("+")
    return c


def _step(sim, act, path):
    if path == "step":
        sim.step(act.tobytes())
    else:
        sim.step(None, half=1)
        sim.step(act.tobytes(), half=2)


class Expected:
    """the tapes of the definition, built from a twin without logs that is stepped half by half: the symbols of a
    step are ind's and those of the slots whose action mask is not 0 between the halves"""

    def __init__(self, name, n):
        self.name, self.ind = name, CONFIGS[name][0].get("ind", 0)
        self.stream, self.steps, self.episode = [b""] * n, [0] * n, [0] * n
        self.status, self.started = [sfcfg.RUNNING] * n, [False] * n

    def step(self, ref, act):
        before = [ref.status(e) for e in range(ref.n_envs)]
        ref.step(None, half=1)
        masks = ref.masks()
        for e in range(ref.n_envs):
            if before[e] != sfcfg.RUNNING:
                continue
            if self.steps[e] == 0:
                self.stream[e], self.started[e] = b"", True
            if ref.status(e) == sfcfg.RUNNING:
                syms = [int(act[e, self.ind])] + [_delivered(self.name, a, int(act[e, a])) for a in range(ref.n_agents)
                                                  if a != self.ind and masks[e, a] != 0]
                self.stream[e] += bytes(syms)
        ref.step(act.tobytes(), half=2)
        ended = []
        for e in range(ref.n_envs):
            if before[e] == sfcfg.RUNNING:
                self.status[e] = ref.step_out(e)["status"]
                self.steps[e] += self.status[e] not in ABORTS  # the arena's count: steps that ran to their end
                if self.status[e] != sfcfg.RUNNING:
                    ended.append(e)
        return ended

    def next_episode(self, e):
        self.steps[e] = 0
        self.episode[e] += 1

    def check(self, rows, e, what):
        h = logcheck.heads(rows[e:e + 1])[0]
        if not self.started[e]:
            assert h["flags"] == 0, what
            return
        tape = logcheck.tape(rows[e])
        want_flags = COMPLETE | (ABORTED if self.status[e] in ABORTS else 0) | (
            UNREPLAYABLE if any(c in JUNK for c in self.stream[e]) else 0)
        got = (int(h["flags"]), int(h["status"]), int(h["steps"]), int(h["level"]), int(h["episode"]),
               int(h["tb"]), int(h["serial"]), int(h["global_id"]), tape)
        want = (want_flags, self.status[e], self.steps[e], _level(self.name, e), self.episode[e],
                common.synth_tb(BASE + e), common.synth_serial(BASE + e, self.episode[e]), BASE + e, self.stream[e])
        assert got == want, "%s arena %d:\n got %s\nwant %s" % (what, e, got, want)


@pytest.mark.parametrize("auto_reset", [True, False], ids=["auto-reset", "reset-finished"])
@pytest.mark.parametrize("path", ["step", "split"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_tapes_equal_the_stream_built_between_the_halves(arena_data, name, path, auto_reset):
    sim, ref = _sim(arena_data, name, auto_reset), _sim(arena_data, name, auto_reset, match_log=0)
    exp = Expected(name, N)
    rng = np.random.default_rng(sum(map(ord, name + path)) + auto_reset)
    ended_total = aborted = agents_logged = 0
    for t in range(STEPS):
        act = _actions(rng, N, sim.n_agents)
        ended = exp.step(ref, act)
        _step(sim, act, path)
        rows = sim.logs()
        for e in range(N):
            exp.check(rows, e, "%s %s step %d" % (name, path, t))
        agents_logged += sum(len(s) for s in exp.stream)
        ended_total += len(ended)
        aborted += sum(exp.status[e] in ABORTS for e in ended)
        for e in ended:
            exp.next_episode(e)
        if not auto_reset:
            sim.reset_finished()
            ref.reset_finished()
    assert ended_total >= N and agents_logged
    if name != "royale16":
        assert aborted, "no episode ended in an abort"


def _oracle_replay(arena_data, name, row, hashes, tmp_path):
    """write the row as a file, read it back and replay it on the C oracle: the recorded hash after every step and
    the final status.  Returns the number of steps replayed."""
    kw = CONFIGS[name][0]
    cfg = _cfg(arena_data, name, False, n=1)
    path = str(tmp_path / ("%s.sf_sample" % name))
    level = replay.write_device_log(path, row, cfg)
    h = logcheck.heads(row[None])[0]
    royale = kw["mode"] == sfcfg.MODE_ROYALE
    if royale:
        log = replay.read_royale(path)
        assert (log.ind, log.teams) == (kw["ind"], kw["teams"])
        ocfg = sfcfg.make_config(arena_data, mode=sfcfg.MODE_ROYALE, teams=log.teams, sheets=list(log.sheets),
                                 ind=log.ind, caps=kw["caps"], max_steps=MAX_STEPS_HERE)
    else:
        log = replay.read(path)
        assert (log.sheet == replay.logged_sheet(list(cfg.player_sheet))).all()
        okw = {k: v for k, v in kw.items() if k not in ("level_min", "level_max")}
        ocfg = sfcfg.make_config(arena_data, level_min=level, max_steps=MAX_STEPS_HERE, **okw)
    assert (log.tb, log.serial, log.commands) == (int(h["tb"]), int(h["serial"]), logcheck.tape(row))
    o = sfo.Arena(ocfg)
    o.reset(level, log.tb, log.serial)
    n_agents = 16 if royale else (10 if kw.get("squad_agents") else 1)
    ind = kw.get("ind", 0)
    pos, status = 0, sfcfg.RUNNING
    for t, want in enumerate(hashes):
        status = o.step_a()
        if status == sfcfg.RUNNING:
            rec = sfo.parse_record(o.dump())
            logged = [ind] + [a for a in range(n_agents) if a != ind and (3, a) in rec and rec[(3, a)][0]
                              and not rec[(3, a)][1]]
            row_a = bytearray(b"+" * n_agents)
            for a in logged:
                row_a[a] = log.commands[pos]
                pos += 1
            status = o.step_b(bytes(row_a))
        if status not in ABORTS:  # the state an abort leaves is undefined; its status is compared below
            assert o.state_hash() == want, "%s step %d: the replay left the recorded episode" % (name, t)
    assert pos == len(log.commands) and status == int(h["status"])
    return len(hashes)


@pytest.mark.parametrize("name", list(CONFIGS))
def test_complete_tapes_replay_on_the_oracle(arena_data, name, tmp_path):
    """auto_reset = 0 and sf_reset_finished, so that the state hash of every step of an episode can be recorded"""
    sim = _sim(arena_data, name, False, n=8)
    rng = np.random.default_rng(3 + len(name))
    hashes = [[] for _ in range(sim.n_envs)]
    replayed = episodes = 0
    for t in range(200):
        running = [sim.status(e) == sfcfg.RUNNING for e in range(sim.n_envs)]
        sim.step(_actions(rng, sim.n_envs, sim.n_agents).tobytes())
        rows = sim.logs()
        for e in range(sim.n_envs):
            if not running[e]:
                continue
            hashes[e].append(sim.state_hash(e))
            if sim.status(e) != sfcfg.RUNNING:
                flags = int(logcheck.heads(rows[e:e + 1])[0]["flags"])
                if flags & COMPLETE and not flags & UNREPLAYABLE:
                    replayed += _oracle_replay(arena_data, name, rows[e], hashes[e], tmp_path) > 0
                else:
                    with pytest.raises(ValueError):
                        replay.write_device_log(str(tmp_path / "refused.sf_sample"), rows[e], _cfg(arena_data, name, False))
                hashes[e], episodes = [], episodes + 1
        sim.reset_finished()
    assert replayed >= 8 and replayed >= episodes // 2, (replayed, episodes)


@needs_reference
@pytest.mark.parametrize("name,mode,agents", [("solo", sfcfg.MODE_SOLO, False), ("squad-agents", sfcfg.MODE_SQUAD, True)])
def test_reference_reader_replays_a_device_written_file(arena_data, name, mode, agents, tmp_path):
    """the reference's own reader replays a file written from a tape to the oracle's final record (default caps, so
    that nothing overflows)"""
    level = 2
    cfg = sfcfg.make_config(arena_data, n_envs=1, mode=mode, level_min=level, squad_agents=agents, auto_reset=False)
    sim = logcheck.LogSim(cfg, match_log=4096)
    rng = np.random.default_rng(21)
    acts = []
    for t in range(150):
        acts.append(np.frombuffer(sfcfg.ACTIONS9 if agents else sfcfg.ACTIONS28, np.uint8)[
            rng.integers(9 if agents else 28, size=(1, sim.n_agents))])
        sim.step(acts[-1].tobytes())
        if sim.status(0) != sfcfg.RUNNING:
            break
    path = str(tmp_path / "device.sf_sample")
    assert replay.write_device_log(path, sim.logs()[0], cfg) == level
    caps = [sfcfg.DEFAULT_CAPS[k] for k in ("cap_humans", "cap_zombies", "cap_bullets", "cap_chests", "cap_built",
                                            "cap_portals")]
    sfref.reset_replay(mode, level, path, squad_agents=agents, caps=caps)
    for t in range(len(acts)):
        if sfref.step(b"+" * sim.n_agents) != 0:
            break
    o = sfo.Arena(sfcfg.make_config(arena_data, mode=mode, level_min=level, squad_agents=agents))
    log = replay.read(path)
    o.reset(level, log.tb, log.serial)
    for a in acts:
        if o.step(a.tobytes()) != 0:
            break
    d0, d1 = sfref.dump(), o.dump()
    assert len(d0) == len(d1) and (d0 == d1).all(), sfo.diff_records(d0, d1)


@pytest.mark.parametrize("tb,serial", [
    (12345, 678), (987654321, 1073741823), (123456789012345, 10 ** 11 + 7), (10 ** 17 + 5, 999999999999999999),
    (1700000000, 123456789), (1771155561, 1073741823), (0, 0)])
def test_seeds_round_trip(arena_data, tb, serial):
    """sf_reset seeds below and above 10^10 and the known-answer seeds come back exactly; the synthetic chain is
    covered by test_tapes_equal_the_stream_built_between_the_halves"""
    sim = _sim(arena_data, "solo", False, n=2)
    sim.reset(1, tb, serial)
    sim.step(b"++")
    h = logcheck.heads(sim.logs())
    assert (int(h[1]["tb"]), int(h[1]["serial"])) == (tb, serial)
    assert (int(h[0]["tb"]), int(h[0]["serial"])) == (common.synth_tb(BASE), common.synth_serial(BASE, 0))


def test_seeds_beyond_18_digits_seed_the_same_stream(arena_data):
    """sf_reset accepts seeds up to 2^63 - 1, of which only 18 digits count: the header carries the seeds modulo
    10^18, and an arena reset with those follows the same stream"""
    tb, serial = 9 * 10 ** 18 + 1700000000, 10 ** 18 + 42
    sim, twin = _sim(arena_data, "solo", False, n=1), _sim(arena_data, "solo", False, n=1, match_log=0)
    sim.reset(0, tb, serial)
    sim.step(b"+")
    h = logcheck.heads(sim.logs())[0]
    assert (int(h["tb"]), int(h["serial"])) == (tb % 10 ** 18, serial % 10 ** 18)
    twin.reset(0, int(h["tb"]), int(h["serial"]))
    twin.step(b"+")
    rng = np.random.default_rng(0)
    for _ in range(30):
        a = bytes(_actions(rng, 1, 1)[0])
        sim.step(a)
        twin.step(a)
        assert sim.state_hash(0) == twin.state_hash(0)


def test_load_clears_complete(arena_data):
    sim = _sim(arena_data, "squad-agents", False, n=4)
    rng = np.random.default_rng(1)
    for _ in range(3):
        sim.step(_actions(rng, 4, sim.n_agents).tobytes())
    assert (logcheck.heads(sim.logs())["flags"] & COMPLETE).all()
    rec = sim.save(2)
    assert sim.load(1, rec)
    assert list(logcheck.heads(sim.logs())["flags"] & COMPLETE) == [COMPLETE, 0, COMPLETE, COMPLETE]
    bad = rec.copy()
    bad[:4] ^= 0xFF
    assert not sim.load(0, bad)  # refused: nothing changes
    assert int(logcheck.heads(sim.logs())[0]["flags"]) & COMPLETE
    recs = np.stack([sim.save(3), bad])
    assert sim.load_list(recs, [0, 3], rows=[0, 1]) == 1  # refused: no tape changes
    assert list(logcheck.heads(sim.logs())["flags"] & COMPLETE) == [COMPLETE, 0, COMPLETE, COMPLETE]
    assert sim.load_list(recs, [0, -1, 0, 4], rows=[0, 1, 1, 1]) == 0  # accepted: the owner of 0 loads
    assert list(logcheck.heads(sim.logs())["flags"] & COMPLETE) == [0, 0, COMPLETE, COMPLETE]
    # a loaded arena whose next step begins an episode restarts its tape
    for _ in range(MAX_STEPS_HERE + 2):
        sim.step(_actions(rng, 4, sim.n_agents).tobytes())
        sim.reset_finished()
    assert (logcheck.heads(sim.logs())["flags"] & COMPLETE).all()


def test_truncated_when_the_tape_is_full(arena_data):
    sim = _sim(arena_data, "squad-agents", False, n=2, match_log=25)
    assert sim.row_bytes == sfcfg.log_row_bytes(25) == 48 + 32
    rng = np.random.default_rng(2)
    full = _sim(arena_data, "squad-agents", False, n=2)
    for _ in range(5):
        a = _actions(rng, 2, sim.n_agents).tobytes()
        sim.step(a)
        full.step(a)
    h, hf = logcheck.heads(sim.logs()), logcheck.heads(full.logs())
    assert (hf["n_symbols"] > 25).all()
    assert (h["n_symbols"] == 25).all() and (h["flags"] == TRUNCATED).all() and (h["steps"] == hf["steps"]).all()
    assert all(logcheck.tape(r) == logcheck.tape(f)[:25] for r, f in zip(sim.logs(), full.logs()))
    with pytest.raises(ValueError):
        replay.write_device_log("/dev/null", sim.logs()[0], _cfg(arena_data, "squad-agents", False))


def test_junk_bytes_are_unreplayable(arena_data, tmp_path):
    """junk bytes reach ind and the Battle Royale players as they are; white space and NUL are flagged"""
    sim = _sim(arena_data, "royale16", False, n=len(JUNK) + 1)
    act = np.full((sim.n_envs, sim.n_agents), ord("+"), np.uint8)
    act[:len(JUNK), 5] = list(JUNK)
    act[len(JUNK), 7] = 0xA0  # not white space for `file >> char`
    sim.step(act.tobytes())
    h = logcheck.heads(sim.logs())
    assert (h["flags"][:len(JUNK)] == COMPLETE | UNREPLAYABLE).all() and h["flags"][-1] == COMPLETE
    assert logcheck.tape(sim.logs()[0])[0] == 0
    with pytest.raises(ValueError):
        replay.write_device_log(str(tmp_path / "junk.sf_sample"), sim.logs()[0], _cfg(arena_data, "royale16", False))


def test_aborted_episodes_are_flagged(arena_data):
    """tiny capacities overflow: the tape says so, and its final status is the abort"""
    sim = _sim(arena_data, "solo", False, n=8)
    rng = np.random.default_rng(4)
    seen = 0
    for _ in range(200):
        running = [sim.status(e) == sfcfg.RUNNING for e in range(8)]
        sim.step(_actions(rng, 8, 1).tobytes())
        h = logcheck.heads(sim.logs())
        for e in range(8):
            st = sim.status(e)
            if running[e] and st in ABORTS:
                assert h[e]["flags"] & ABORTED and h[e]["status"] == st
                seen += 1
            elif running[e]:
                assert not h[e]["flags"] & ABORTED
        sim.reset_finished()
    assert seen


@pytest.mark.parametrize("name", list(CONFIGS))
def test_list_step_appends_for_listed_arenas_only(arena_data, name):
    """a list step appends for each id's owning entry and leaves unlisted tapes alone; S then its complement gives
    the tapes of one whole step"""
    whole, parts = _sim(arena_data, name, True), _sim(arena_data, name, True)
    rng = np.random.default_rng(sum(map(ord, name)))
    for t in range(150):
        act = _actions(rng, N, whole.n_agents)
        whole.step(act.tobytes())
        inside = rng.random(N) < rng.random()
        for part in (np.nonzero(inside)[0], np.nonzero(~inside)[0]):
            prev = parts.logs()
            dup = rng.choice(part, size=min(len(part), 2)) if len(part) else np.zeros(0, int)
            ids = np.concatenate([rng.permutation(part), dup, [-1, N]]).astype(np.int32)
            rows = np.full((len(ids), whole.n_agents), ord("_"), np.uint8)  # the repeats must not step
            rows[:len(part)] = act[ids[:len(part)]]
            parts.step_list(rows, ids)
            out = np.setdiff1d(np.arange(N), part)
            assert (parts.logs()[out] == prev[out]).all(), "%s step %d: an unlisted tape changed" % (name, t)
        assert (parts.logs() == whole.logs()).all(), "%s step %d" % (name, t)


@pytest.mark.parametrize("path", ["step", "split"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_logs_change_nothing_else(arena_data, name, path):
    """logs and agent outputs on against agent outputs alone, and logs alone against nothing: state hashes,
    sf_step_out, agent rows, statistics and records"""
    both, ao = _sim(arena_data, name, True, agent_out=True), _sim(arena_data, name, True, agent_out=True, match_log=0)
    logs, off = _sim(arena_data, name, True), _sim(arena_data, name, True, match_log=0)
    rng = np.random.default_rng(13)
    for t in range(200):
        act = _actions(rng, N, both.n_agents)
        for s in (both, ao, logs, off):
            _step(s, act, path)
        assert (both.agent_out() == ao.agent_out()).all(), "%s %s step %d" % (name, path, t)
        for e in range(N):
            h = off.state_hash(e)
            assert both.state_hash(e) == ao.state_hash(e) == logs.state_hash(e) == h, "%s %s step %d" % (name, path, t)
            assert both.step_out(e) == ao.step_out(e) == logs.step_out(e) == off.step_out(e)
    assert (both.logs() == logs.logs()).all()
    assert both.stats() == ao.stats() == logs.stats() == off.stats()
    for e in range(N):
        assert (both.save(e) == off.save(e)).all() and (logs.save(e) == off.save(e)).all()


def test_enable_log_arguments(arena_data):
    sim = _sim(arena_data, "solo", False, n=2, match_log=0)
    assert not sim.enable_log(0) and not sim.enable_log(sfcfg.LOG_CAP_MAX + 1)
    assert sim.enable_log(100) and sim.enable_log(100) and not sim.enable_log(101)
    assert sim.row_bytes == sfcfg.log_row_bytes(100) == 48 + 112


def test_header_mirrors_config():
    """SF_LOG_* and the fields of sf_log_head equal the Python mirror"""
    text = open(os.path.join(ROOT, "include", "strikeforce_b200.h")).read()
    for name in ("COMPLETE", "TRUNCATED", "ABORTED", "UNREPLAYABLE"):
        assert int(re.search(r"SF_LOG_%s\s*=\s*(\d+)" % name, text).group(1)) == getattr(sfcfg, "LOG_" + name)
    assert re.search(r"#define SF_LOG_CAP_MAX \(1 << (\d+)\)", text).group(1) == "24" and sfcfg.LOG_CAP_MAX == 1 << 24
    body = re.search(r"typedef struct sf_log_head \{(.*?)\} sf_log_head;", text, re.S).group(1)
    fields = re.findall(r"(u?int\d+)_t\s+(\w+)(?:,\s*(\w+))?;", body)
    names = [n for _, a, b in fields for n in (a, b) if n]
    assert tuple(names) == sfcfg.LOG_HEAD.names
    size = {"int32": 4, "uint32": 4, "int64": 8}
    assert [size[t] for t, a, b in fields for n in (a, b) if n] == [sfcfg.LOG_HEAD[n].itemsize for n in names]
