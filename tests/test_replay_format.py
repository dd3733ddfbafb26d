"""The .sf_sample log (SURVEY 8f rank 1): strikeforce_b200/replay.py against the reference's OWN
writer (enable_logging) and reader (replay mode), through oracle/_ref."""
import os

import numpy as np
import pytest

import sfo
import sfref
from strikeforce_b200 import config as sfcfg
from strikeforce_b200 import replay

needs_reference = pytest.mark.skipif(not sfref.available(), reason="oracle/_ref/libsfref.so not built")

CAPS = [sfcfg.DEFAULT_CAPS[k] for k in ("cap_humans", "cap_zombies", "cap_bullets", "cap_chests", "cap_built",
                                        "cap_portals")]


@needs_reference
def test_writer_matches_the_reference_logger(arena_data, tmp_path):
    """The reference logs a Solo match; our writer reproduces the file byte for byte, our reader
    recovers seeds, sheet and commands."""
    rng = np.random.default_rng(11)
    tb, serial = sfref.reset_logging(sfcfg.MODE_SOLO, 2, caps=CAPS)
    cmds = bytes(sfcfg.ACTIONS28[i] for i in rng.integers(28, size=120))
    for c in cmds:
        assert sfref.step(bytes([c])) == 0
    path = sfref.close_log()
    ref_bytes = open(path, "rb").read()
    os.remove(path)
    ours = tmp_path / "ours.sf_sample"
    replay.write(str(ours), tb, serial, replay.logged_sheet(arena_data.player_sheet("account1")), cmds)
    assert open(ours, "rb").read() == ref_bytes
    log = replay.read(str(ours))
    assert (log.tb, log.serial, log.players, log.ind, log.team, log.name) == (tb, serial, 1, 0, 1, "1")
    assert log.commands == cmds
    assert (log.sheet == replay.logged_sheet(arena_data.player_sheet("account1"))).all()


@needs_reference
@pytest.mark.parametrize("mode,level,agents", [(sfcfg.MODE_SOLO, 1, False), (sfcfg.MODE_SQUAD, 2, True)])
def test_reference_replays_our_file_like_the_oracle(arena_data, tmp_path, mode, level, agents):
    """A file written by us is replayed by the reference's own reader; the oracle, fed by our reader,
    follows it state for state."""
    rng = np.random.default_rng(5 + mode)
    sheet = arena_data.player_sheet("new_player").copy()
    sheet[11:15] = [3, 2, 1, 4]
    sheet[16:23:2] = [2, 2, 2, 2]
    sheet[23:31] = [1, 0, 2, 0, 1, 1, 0, 3]
    sheet[3:6] = [3, 2, 4]
    steps, n = 150, (10 if agents else 1)
    table = sfcfg.ACTIONS9 if agents else sfcfg.ACTIONS28
    per_step = [bytes(table[i] for i in rng.integers(len(table), size=n)) for _ in range(steps)]
    path = tmp_path / "match.sf_sample"
    # squad agents may die; the log then simply stops listing them -- keep everyone alive by
    # writing commands for all ten and checking liveness while replaying
    tb, serial = 1700001234, 987654
    cfg = sfcfg.make_config(arena_data, mode=mode, level_min=level, squad_agents=agents, player=sheet)
    o = sfo.Arena(cfg)
    o.reset(level, tb, serial)
    stream = b""
    for t in range(steps):
        # the log lists the humans that are alive when human_action runs, i.e. after half-tick A
        if o.step_a() != 0:
            steps = t
            break
        alive = [0] + [h for h in range(1, n) if sfo.parse_record(o.dump())[(3, h)][0]]
        stream += bytes(per_step[t][h] for h in alive)
        if o.step_b(per_step[t]) != 0:
            steps = t + 1
            break
    replay.write(str(path), tb, serial, sheet, stream, name="tester")
    log = replay.read(str(path))
    assert log.commands == stream and (log.sheet == sheet).all()
    sfref.reset_replay(mode, level, str(path), squad_agents=agents, caps=CAPS)
    o.reset(level, log.tb, log.serial)
    d0, d1 = sfref.dump(), o.dump()
    assert len(d0) == len(d1) and (d0 == d1).all(), sfo.diff_records(d0, d1)
    for t in range(steps):
        s0 = sfref.step(b"+" * n)  # the reference takes every command from the file
        s1 = o.step(per_step[t])
        assert s0 == s1, "status, step %d" % t
        if s0 != 0:
            break
        d0, d1 = sfref.dump(), o.dump()
        assert len(d0) == len(d1) and (d0 == d1).all(), "step %d: %s" % (t, sfo.diff_records(d0, d1))


def test_royale_log_round_trip(tmp_path, arena_data):
    """write_royale -> read_royale: the online replay format (gameplay.hpp:1762-1806) has a reader too."""
    import pytest
    from strikeforce_b200 import replay
    rng = np.random.default_rng(9)
    teams = [2, 1, 3, 1, 2]
    sheets = np.stack([np.asarray(arena_data.player_sheet("account1"), dtype=np.int32) + i for i in range(5)])
    cmds = bytes(sfcfg.ACTIONS28[j] for j in rng.integers(28, size=97))
    path = tmp_path / "online.sf_sample"
    replay.write_royale(str(path), 1700000321, 987654, sheets, teams, cmds, ind=2)
    log = replay.read_royale(str(path))
    assert (log.tb, log.serial, log.ind, log.teams) == (1700000321, 987654, 2, teams)
    assert (log.sheets == sheets).all() and log.commands == cmds and log.names[2] == "player2"
    with pytest.raises(ValueError):
        replay.read(str(path))  # the offline reader refuses it instead of folding sheets into commands
