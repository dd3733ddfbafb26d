"""ctypes mirror of ``include/strikeforce_b200.h`` (struct layouts, enums) and the builder of
an ``sf_config`` from :class:`strikeforce_b200.data.ArenaData`.

``sf_config`` replaces what the reference takes from its menus and data files:
mode / level prompts of ``gameplay::open`` (gameplay.hpp:1507-1678), ``map/``, ``Items/``,
``character/`` and the account sheet (gameplay.hpp:1231-1277, Item.hpp:179-188,
Character.hpp:650-709).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import data as sfdata

ABI_VERSION = 3
# SF_FLOORS / SF_ROWS / SF_COLS (gameplay.hpp:37); SF_GEOMETRY in the environment selects a larger arena (data.py)
FLOORS, ROWS, COLS = sfdata.FLOORS, sfdata.ROWS, sfdata.COLS
CELLS = FLOORS * ROWS * COLS
GEOMETRY_TAG, GEOMETRY_CFLAGS = sfdata.GEOMETRY_TAG, sfdata.GEOMETRY_CFLAGS
OBS_CH, OBS_WIN = 32, 31
OBS_LEN = OBS_CH * OBS_WIN * OBS_WIN
SHEET_LEN = sfdata.SHEET_LEN

MODE_SOLO, MODE_TIMER, MODE_SQUAD, MODE_ROYALE = 0, 1, 2, 3
MODES = {"Solo": MODE_SOLO, "Timer": MODE_TIMER, "Squad": MODE_SQUAD, "Royale": MODE_ROYALE, "Battle Royal": MODE_ROYALE}
MAX_PLAYERS = 16

RUNNING, WIN, DEAD, TIMEOUT, TRUNCATED, OVERFLOW, UB_GUARD = range(7)
STATUS_NAMES = ["running", "win", "dead", "timeout", "truncated", "overflow", "ub_guard"]

OBS_P1, OBS_P2 = 1, 2
OBS_NHWC = 0x100  # OR-ed into the phase: channel innermost
OBS_F16, OBS_BF16 = 0x200, 0x400  # OR-ed into the phase (at most one): fp16 / bfloat16 values, rounded to nearest even

FIELD_STEP_OUT, FIELD_STATE_HASH, FIELD_COUNTERS, FIELD_POPULATION, FIELD_STATS = 1, 2, 3, 4, 5
FIELD_AGENT_OUT = 6  # sf_agent_out [n_envs][n_agents], after sf_enable_agent_out
# sf_agent_out: the per-agent step outputs (include/strikeforce_b200.h, DESIGN.md section 7g)
AGENT_DRIVEN, AGENT_DIED = 1, 2  # bits of the flags field
AGENT_OUT_FIELDS = ("flags", "d_hp", "d_damage", "d_effect", "d_kills")
# match logs (sf_enable_log / sf_log_list, include/strikeforce_b200.h, DESIGN.md section 7h)
LOG_COMPLETE, LOG_TRUNCATED, LOG_ABORTED, LOG_UNREPLAYABLE = 1, 2, 4, 8  # bits of the flags field
LOG_CAP_MAX = 1 << 24
# sf_log_head, the start of an exported row; cap_symbols bytes of tape follow, the row padded to 16 bytes
LOG_HEAD = np.dtype([("flags", "<i4"), ("status", "<i4"), ("level", "<i4"), ("episode", "<u4"), ("steps", "<i4"),
                     ("n_symbols", "<i4"), ("tb", "<i8"), ("serial", "<i8"), ("global_id", "<i8")])


def log_row_bytes(cap_symbols):
    """bytes of one exported row (sf_log_row_bytes)"""
    return LOG_HEAD.itemsize + (cap_symbols + 15) // 16 * 16


# replay (sf_enable_replay / sf_replay_load, include/strikeforce_b200.h, DESIGN.md section 7i)
FIELD_REPLAY = 7        # sf_replay_state [n_envs], after sf_enable_replay
FIELD_REPLAY_DEALT = 8  # uint8 [n_envs][n_agents]: the symbols the last step took from the tapes
REPLAY_ARMED, REPLAY_EXHAUSTED, REPLAY_ENDED, REPLAY_SURPLUS = 1, 2, 4, 8  # bits of the flags field
REPLAY_STATE = np.dtype([("flags", "<i4"), ("cursor", "<i4"), ("n_symbols", "<i4"), ("steps", "<i4"), ("status", "<i4")])


def replay_row_bytes(cap_symbols):
    """bytes of one load row (sf_replay_row_bytes): the layout of an exported match-log row"""
    return log_row_bytes(cap_symbols)


STAT_NAMES = ["steps", "episodes", "wins", "deaths", "timeouts", "truncated", "overflows", "ub_guards",
              "kills", "teams_kills", "loot", "rng_draws", "algo_bytes", "reserved0", "reserved1", "reserved2"]

# valid_commands (gameplay.hpp:45) and the 9 symbols the shipped bots expose (Custom.hpp:162)
ACTIONS9 = b"+xzqeawsd"
ACTIONS28 = b"+qeuzxawsdfghjkl;'cvbnm,./[]"
# SF_COMMANDS: the alphabet of sf_action_mask in bit order (valid_commands, then '_'); bit j stands for COMMANDS[j]
COMMANDS = b"+qe3uzxawsdfghjkl;'cvbnm,./[]_"
N_COMMANDS = 30

ERRORS = {0: "ok", -1: "bad argument", -2: "no CUDA device (there is no CPU path)", -3: "CUDA error",
          -4: "unsupported", -5: "out of memory"}


class Consumable(C.Structure):
    _fields_ = [("stamina", C.c_int32), ("hp", C.c_int32), ("effect", C.c_int32)]


class Weapon(C.Structure):
    _fields_ = [("stamina", C.c_int32), ("damage", C.c_int32), ("effect", C.c_int32), ("range", C.c_int32)]


class SfConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("n_envs", C.c_int32),
        ("env_id_base", C.c_int64),
        ("mode", C.c_int32),
        ("level_min", C.c_int32),
        ("level_max", C.c_int32),
        ("squad_agents", C.c_int32),
        ("auto_reset", C.c_int32),
        ("max_steps", C.c_int32),
        ("cap_humans", C.c_int32),
        ("cap_zombies", C.c_int32),
        ("cap_bullets", C.c_int32),
        ("cap_chests", C.c_int32),
        ("cap_built", C.c_int32),
        ("cap_portals", C.c_int32),
        ("map_cells", C.POINTER(C.c_uint8)),
        ("map_portal", C.POINTER(C.c_int16)),
        ("consumables", Consumable * 4),
        ("throwables", Weapon * 4),
        ("weapons", Weapon * 8),
        ("player_sheet", C.c_int32 * SHEET_LEN),
        ("npc_sheet", C.c_int32 * SHEET_LEN),
        ("royale_players", C.c_int32),
        ("royale_teams", C.c_int32 * MAX_PLAYERS),
        ("royale_sheets", (C.c_int32 * SHEET_LEN) * MAX_PLAYERS),
        ("royale_ind", C.c_int32),
    ]


class StepOut(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("status", "d_kills", "d_teams_kills", "d_loot", "d_hp", "d_damage", "d_effect", "episode_steps")]


STEP_OUT_DTYPE = np.dtype([(n, np.int32) for n, _ in StepOut._fields_])

DEFAULT_CAPS = dict(cap_humans=64, cap_zombies=128, cap_bullets=96, cap_chests=9000, cap_built=384, cap_portals=96)


def make_config(arena: sfdata.ArenaData, n_envs=1, mode=MODE_SOLO, level_min=1, level_max=None, squad_agents=False,
                auto_reset=True, max_steps=0, env_id_base=0, player="account1", caps=None, teams=None, sheets=None, ind=0):
    """Build an ``sf_config``.  The returned struct keeps the numpy arrays it points to alive
    (``cfg._keep``).  Battle Royale only: ``teams`` = the team of each player, e.g. ``[1, 1, 2, 2]``;
    ``sheets`` = the character sheet of each player (names or int32[32] arrays; default: every
    player carries ``player``; entry ``ind`` is the sheet of ``ind`` and replaces ``player``); ``ind`` = the
    player whose copy of the match the arenas are (credits, the corpse that keeps its cell, the end of the match)."""
    if isinstance(mode, str):
        mode = MODES[mode]
    cfg = SfConfig()
    cfg.abi_version = ABI_VERSION
    cfg.n_envs = n_envs
    cfg.env_id_base = env_id_base
    cfg.mode = mode
    cfg.level_min = level_min
    cfg.level_max = level_min if level_max is None else level_max
    cfg.squad_agents = int(bool(squad_agents))
    cfg.auto_reset = int(bool(auto_reset))
    cfg.max_steps = max_steps
    c = dict(DEFAULT_CAPS)
    c.update(caps or {})
    for k, v in c.items():
        setattr(cfg, k, v)
    cells = np.ascontiguousarray(arena.map_cells, dtype=np.uint8)
    portal = np.ascontiguousarray(arena.map_portal, dtype=np.int16)
    cfg.map_cells = cells.ctypes.data_as(C.POINTER(C.c_uint8))
    cfg.map_portal = portal.ctypes.data_as(C.POINTER(C.c_int16))
    for i in range(4):
        cfg.consumables[i] = Consumable(*[int(v) for v in arena.consumables[i]])
        cfg.throwables[i] = Weapon(*[int(v) for v in arena.throwables[i]])
    for i in range(8):
        cfg.weapons[i] = Weapon(*[int(v) for v in arena.weapons[i]])
    def as_sheet(x):
        return arena.player_sheet(x) if isinstance(x, str) else np.asarray(x, dtype=np.int32)

    if mode == MODE_ROYALE and sheets is not None:
        player = sheets[ind]
    sheet = as_sheet(player)
    for i in range(SHEET_LEN):
        cfg.player_sheet[i] = int(sheet[i])
        cfg.npc_sheet[i] = int(arena.npc_sheet[i])
    if mode == MODE_ROYALE:
        teams = list(teams if teams is not None else [1 + i % 4 for i in range(MAX_PLAYERS)])
        if not 2 <= len(teams) <= MAX_PLAYERS:
            raise ValueError("Battle Royale needs 2..%d players" % MAX_PLAYERS)
        cfg.royale_players = len(teams)
        if sheets is not None and len(sheets) != len(teams):
            raise ValueError("one sheet per player")
        for i, t in enumerate(teams):
            cfg.royale_teams[i] = int(t)
            sh = sheet if sheets is None else as_sheet(sheets[i])
            for j in range(SHEET_LEN):
                cfg.royale_sheets[i][j] = int(sh[j])
        if not 0 <= ind < len(teams):
            raise ValueError("ind must name one of the players")
        cfg.royale_ind = ind
        cfg.level_min = cfg.level_max = 1  # gameplay.hpp:1641, 1659
    cfg._keep = (cells, portal)
    return cfg


def dump_config(cfg: SfConfig, path):
    """Write ``cfg`` as the blob the C++ host reads (strikeforce_b200/host/bot-b200/Custom.hpp,
    ``sfb200::Config::load``): the struct as it lies in memory, then map_cells[CELLS] (uint8), then
    map_portal[CELLS] (int16).  The two pointers inside the struct are meaningless in the file."""
    cells = np.ctypeslib.as_array(cfg.map_cells, shape=(CELLS,)).astype(np.uint8)
    portal = np.ctypeslib.as_array(cfg.map_portal, shape=(CELLS,)).astype(np.int16)
    with open(path, "wb") as f:
        f.write(bytes(cfg))
        f.write(cells.tobytes())
        f.write(portal.tobytes())
