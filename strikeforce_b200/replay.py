"""The reference's ``.sf_sample`` match log (SURVEY.md 8f, rank 1): read and write.

Format, as written by ``gameplay::load_data`` / ``human_action`` with ``enable_logging``
(gameplay.hpp:1864-1870, 1909-1914, 966-967, 982-991) and read back in replay mode
(:1771-1783, 968-993; ``Human::scan_file`` / ``log_file`` Character.hpp:570-648), offline modes::

    <tb> <serial>                      seeds of Random::_srand
    <players> <ind> <team>             "1 0 1" offline
    <name>                             the player's character sheet, one value per line:
    <def_Hp> <mindamage_def> <def_stamina> <level_solo> <level_timer> <level_squad> <money>
    <rate_solo> <rate_timer> <rate_squad> <rate> <cons x4> <(throw level, count) x4>
    <weapon level x8> <backpack level>
    <command>                          then one symbol per line: the player's command of the step,
    <command> ...                      followed by that of every agent-driven squad human that is
                                       alive when human_action runs, i.e. after the first half-tick
                                       (ascending slot), when USE_AGENT_IN_SQUAD_NPCS is on

Two quirks of the reference are part of the format: the sheet is logged AFTER the account's own
level-ups were applied to the three ``def_*`` values (``log_file`` writes the live fields), and the
reader applies them again (``scan_file``); and the reader takes its seeds from the file, so a log
replays deterministically.  ``logged_sheet`` computes what the reference writes for an account
sheet; ``read`` returns exactly what the reference's reader would consume.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import data as sfdata


@dataclass
class MatchLog:
    tb: int
    serial: int
    players: int
    ind: int
    team: int
    name: str
    sheet: np.ndarray  # int32 [32], as stored in the file
    commands: bytes  # the command symbols in file order


def logged_sheet(sheet):
    """The sheet values ``Human::log_file`` writes for a character built from ``sheet``
    (Human::build applies level-1 ups per mode to def_Hp / mindamage_def / def_stamina,
    Character.hpp:690-708, 765-801)."""
    s = np.array(sheet, dtype=np.int32).copy()
    ups = int(sum(max(int(l) - 1, 0) for l in s[3:6]))
    s[0] += 50 * ups
    s[1] += 5 * ups
    s[2] += 50 * ups
    return s


def write(path, tb, serial, sheet, commands, name="1", players=1, ind=0, team=1):
    """Write a log.  ``sheet`` is stored as given (use ``logged_sheet`` to mimic the reference's
    logger); ``commands`` is the byte string of symbols in file order."""
    sheet = np.asarray(sheet, dtype=np.int64)
    assert sheet.shape == (sfdata.SHEET_LEN,)
    with open(path, "w") as f:
        f.write("%d %d\n" % (tb, serial))
        f.write("%d %d %d\n" % (players, ind, team))
        f.write(name + "\n")
        for v in sheet:
            f.write("%d\n" % int(v))
        for c in bytes(commands):
            f.write(chr(c) + "\n")


def write_royale(path, tb, serial, sheets, teams, commands, ind=0):
    """A Battle Royale match as the reference's replay reader takes it (gameplay.hpp:1762-1806): the
    three tokens of the server line, the seeds, ``players ind team``, the sheet of ``ind``, then sheet
    and team of every other player in slot order; ``commands`` are the symbols in file order -- each
    step the command of ``ind``, then that of every other player alive when human_action runs
    (ascending slot, :966-986).  ``sheets``: one int32[32] sheet per player, or a single sheet for all."""
    sheets = np.asarray(sheets, dtype=np.int64)
    if sheets.ndim == 1:
        sheets = np.tile(sheets, (len(teams), 1))
    assert sheets.shape == (len(teams), sfdata.SHEET_LEN) and 2 <= len(teams)
    with open(path, "w") as f:
        f.write("127.0.0.1 0 none\n")
        f.write("%d %d\n" % (tb, serial))
        f.write("%d %d %d\n" % (len(teams), ind, teams[ind]))
        for i in [ind] + [j for j in range(len(teams)) if j != ind]:
            f.write("player%d\n" % i)
            for v in sheets[i]:
                f.write("%d\n" % int(v))
            if i != ind:
                f.write("%d\n" % teams[i])
        for c in bytes(commands):
            f.write(chr(c) + "\n")


@dataclass
class RoyaleLog:
    server: tuple       # the three tokens of the server line (ip, port, password)
    tb: int
    serial: int
    ind: int
    teams: list          # team of every player, slot order
    names: list
    sheets: np.ndarray   # int32 [players, 32], slot order, as stored in the file
    commands: bytes      # the command symbols in file order


def read_royale(path):
    """The reader of ``write_royale``: an online match as the reference's replay mode consumes it
    (gameplay.hpp:1762-1806) -- the server line, the seeds, ``players ind team``, the sheet of ``ind``,
    then sheet and team of every other player in slot order, then the commands."""
    with open(path, "rb") as f:
        tok = f.read().decode("latin-1").split()
    server = tuple(tok[:3])
    tb, serial, players, ind, team = (int(t) for t in tok[3:8])
    if not (2 <= players <= 64 and 0 <= ind < players):
        raise ValueError("%s: not an online match log (players %d, ind %d)" % (path, players, ind))
    pos = 8
    names, sheets, teams = [None] * players, np.zeros((players, sfdata.SHEET_LEN), dtype=np.int32), [0] * players
    for i in [ind] + [j for j in range(players) if j != ind]:
        names[i] = tok[pos]
        sheets[i] = [int(t) for t in tok[pos + 1:pos + 1 + sfdata.SHEET_LEN]]
        pos += 1 + sfdata.SHEET_LEN
        if i == ind:
            teams[i] = team
        else:
            teams[i] = int(tok[pos])
            pos += 1
    return RoyaleLog(server, tb, serial, ind, teams, names, sheets, "".join(tok[pos:]).encode("latin-1"))


def read(path):
    """Parse an OFFLINE log the way the reference's stream extraction does (whitespace separated
    tokens; every command is one non-blank character).  Online match files start with the server
    line and are read by ``read_royale``."""
    with open(path, "rb") as f:
        text = f.read().decode("latin-1")
    tok = text.split()
    if not tok[0].lstrip("-").isdigit():
        raise ValueError("%s starts with %r: an online match log, use read_royale" % (path, tok[0]))
    tb, serial, players, ind, team = (int(t) for t in tok[:5])
    name = tok[5]
    sheet = np.array([int(t) for t in tok[6:6 + sfdata.SHEET_LEN]], dtype=np.int32)
    rest = "".join(tok[6 + sfdata.SHEET_LEN:])  # `file >> char` skips blanks, so tokens simply concatenate
    return MatchLog(tb, serial, players, ind, team, name, sheet, rest.encode("latin-1"))


def write_device_log(path, row, cfg, name="1"):
    """Write the match-log row ``row`` (one row of ``BatchedArena.match_logs()`` on the host: uint8 numpy array or
    bytes) of a handle created with configuration ``cfg`` (``config.make_config``, e.g. ``BatchedArena.cfg``) as a
    ``.sf_sample`` file the reference's replay mode reads.  Offline modes go through ``write`` with the logged
    player sheet, Battle Royale through ``write_royale`` with the handle's teams, sheets and ``ind``.  Returns the
    episode's level, which the offline format does not carry (the client's menu asks for it).

    Raises ValueError for a row that is not ``LOG_COMPLETE`` (a tape that restarted before this handle logged, was
    overwritten by a load, or ran out of capacity) or is ``LOG_UNREPLAYABLE`` (a symbol the reference's reader skips):
    such a file would replay a different episode."""
    from . import config as sfcfg
    row = np.frombuffer(bytes(row), dtype=np.uint8)
    head = row[:sfcfg.LOG_HEAD.itemsize].view(sfcfg.LOG_HEAD)[0]
    flags = int(head["flags"])
    if not flags & sfcfg.LOG_COMPLETE:
        raise ValueError("match log of arena %d is not complete (flags %#x)" % (int(head["global_id"]), flags))
    if flags & sfcfg.LOG_UNREPLAYABLE:
        raise ValueError("match log of arena %d holds a symbol the reference cannot read back" % int(head["global_id"]))
    start = sfcfg.LOG_HEAD.itemsize
    commands = row[start:start + int(head["n_symbols"])].tobytes()
    tb, serial = int(head["tb"]), int(head["serial"])
    if cfg.mode == sfcfg.MODE_ROYALE:
        n = cfg.royale_players
        sheets = np.array([list(cfg.royale_sheets[i]) for i in range(n)], dtype=np.int32)
        write_royale(path, tb, serial, sheets, [cfg.royale_teams[i] for i in range(n)], commands, ind=cfg.royale_ind)
    else:
        write(path, tb, serial, logged_sheet(list(cfg.player_sheet)), commands, name=name)
    return int(head["level"])


def tape_rows(logs, cfg, cap, levels=1):
    """Load rows for ``BatchedArena.replay_load`` (uint8 numpy [len(logs), config.replay_row_bytes(cap)]) from
    ``MatchLog`` / ``RoyaleLog`` objects (``read`` / ``read_royale``) for a handle created with configuration ``cfg``
    and ``replay=cap``.  ``levels``: the level of each offline log, or one level for all (the offline format does not
    carry it); Battle Royale plays level 1.  The head holds the log's seeds, the level, episode 0 and the number of
    symbols.  Rows exported by ``BatchedArena.match_logs()`` are already load rows.

    The device never sees character sheets, so a log the handle cannot replay raises ValueError: an offline log on a
    Battle Royale handle or the reverse, a player sheet, teams, ``ind`` or sheets other than what ``write_device_log``
    writes for ``cfg``, or more symbols than ``cap``."""
    from . import config as sfcfg
    logs = list(logs)
    levels = list(levels) if np.ndim(levels) else [int(levels)] * len(logs)
    assert len(levels) == len(logs)
    rows = np.zeros((len(logs), sfcfg.replay_row_bytes(cap)), dtype=np.uint8)
    royale = cfg.mode == sfcfg.MODE_ROYALE
    for i, (log, level) in enumerate(zip(logs, levels)):
        if royale:
            if not isinstance(log, RoyaleLog):
                raise ValueError("log %d: an offline match log cannot be replayed on a Battle Royale handle" % i)
            n = cfg.royale_players
            sheets = np.array([list(cfg.royale_sheets[j]) for j in range(n)], dtype=np.int32)
            if (log.ind != cfg.royale_ind or list(log.teams) != [cfg.royale_teams[j] for j in range(n)]
                    or log.sheets.shape != sheets.shape or (log.sheets != sheets).any()):
                raise ValueError("log %d: players, ind, teams or sheets differ from the handle's" % i)
            level = 1
        else:
            if not isinstance(log, MatchLog):
                raise ValueError("log %d: a Battle Royale match log needs a Battle Royale handle" % i)
            if (log.players, log.ind, log.team) != (1, 0, 1):
                raise ValueError("log %d: not an offline match of one player (players %d, ind %d, team %d)"
                                 % (i, log.players, log.ind, log.team))
            if (log.sheet != logged_sheet(list(cfg.player_sheet))).any():
                raise ValueError("log %d: the player sheet differs from the handle's" % i)
        if len(log.commands) > cap:
            raise ValueError("log %d: %d symbols do not fit tapes of %d" % (i, len(log.commands), cap))
        head = np.zeros(1, dtype=sfcfg.LOG_HEAD)
        head["level"], head["n_symbols"], head["tb"], head["serial"] = level, len(log.commands), log.tb, log.serial
        rows[i, :sfcfg.LOG_HEAD.itemsize] = head.view(np.uint8)
        rows[i, sfcfg.LOG_HEAD.itemsize:sfcfg.LOG_HEAD.itemsize + len(log.commands)] = np.frombuffer(log.commands, np.uint8)
    return rows


def commands_per_step(log: MatchLog, n_agents_alive):
    """Split the command stream into steps: ``n_agents_alive(step)`` = number of logged humans that
    step (1 offline without squad agents)."""
    out, pos, step = [], 0, 0
    while pos < len(log.commands):
        n = n_agents_alive(step)
        out.append(log.commands[pos:pos + n])
        pos += n
        step += 1
    return out


def drive(sim, logs, steps=None):
    """Replay match logs on a ``BatchedArena`` (one arena per log, same player sheet as the handle
    was created with; offline logs without squad agents).  Returns the per-step status array
    [steps, len(logs)].  The commands never leave the device once uploaded."""
    import torch
    n = len(logs)
    assert n <= sim.n_envs and sim.n_agents == 1
    ids = list(range(n))
    sim.reset(ids, [l.tb for l in logs], [l.serial for l in logs])
    steps = min(len(l.commands) for l in logs) if steps is None else steps
    plan = np.full((steps, sim.n_envs, 1), ord("+"), dtype=np.uint8)
    for e, l in enumerate(logs):
        plan[:, e, 0] = np.frombuffer(l.commands[:steps], dtype=np.uint8)
    plan_d = torch.from_numpy(plan).to(sim.device)
    status = []
    for t in range(steps):
        sim.step(plan_d[t])
        status.append(sim.step_out()[:n, 0].clone())
    return torch.stack(status).cpu().numpy()
