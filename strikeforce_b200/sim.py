"""Host-side driver of the batched simulator: the object a trainer holds instead of the
reference's process-wide ``gameplay g`` (gameplay.hpp:437-1739).

``BatchedArena`` owns one ``sf_handle`` (one GPU).  torch is used for what it is good at here:
device buffers, streams and ``torch.distributed``; all simulation work happens in the CUDA
library behind the C ABI (``strikeforce_b200.lib``).  Tensors handed to / returned from this
class live on the handle's device; nothing round-trips through the host unless the caller
asks for it (``step_host``, ``export_env``).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import config as sfcfg
from . import data as sfdata
from .lib import check, lib


_OBS_FORMAT = {torch.float32: 0, torch.float16: sfcfg.OBS_F16, torch.bfloat16: sfcfg.OBS_BF16}


class BatchedArena:
    def __init__(self, n_envs, mode="Solo", level=1, level_max=None, squad_agents=False, auto_reset=True,
                 max_steps=0, env_id_base=0, player="account1", caps=None, arena=None, device=None, teams=None, sheets=None,
                 ind=0, agent_out=False, match_log=0, replay=0):
        """``agent_out=True`` turns on the per-agent step outputs (sf_enable_agent_out, read with ``agent_out()``)
        from the first step on.  ``match_log`` > 0 turns on match logs (sf_enable_log, read with ``match_logs()``)
        with tapes of that many command symbols.  ``replay`` > 0 turns on replay (sf_enable_replay, loaded with
        ``replay_load()``) with tapes of that many command symbols."""
        if not torch.cuda.is_available():
            # fail loudly: there is no CPU path (sf_create would report SF_ERR_NO_DEVICE as well)
            raise RuntimeError("strikeforce_b200 needs a CUDA device; it has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        torch.cuda.set_device(self.device)
        self.arena = arena or sfdata.load_default()
        self.cfg = sfcfg.make_config(self.arena, n_envs=n_envs, mode=mode, level_min=level, level_max=level_max,
                                     squad_agents=squad_agents, auto_reset=auto_reset, max_steps=max_steps,
                                     env_id_base=env_id_base, player=player, caps=caps, teams=teams, sheets=sheets, ind=ind)
        self._h = C.c_void_p()
        check(lib().sf_create(C.byref(self.cfg), C.byref(self._h)))
        self.n_envs = n_envs
        self.n_agents = lib().sf_agents_per_env(self._h)
        self.step_count = 0
        self._synth = torch.empty((n_envs, self.n_agents), dtype=torch.uint8, device=self.device)
        self._mask_bits = {}  # action_mask(table=): bit index of each symbol of a table, on the device
        if agent_out:
            self._chk(lib().sf_enable_agent_out(self._h))
        if match_log:
            self._chk(lib().sf_enable_log(self._h, match_log))
        if replay:
            self._chk(lib().sf_enable_replay(self._h, replay))

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().sf_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _chk(self, rc):
        check(rc, self._h)

    # ------------------------------------------------------------------ reset / step
    def reset(self, env_ids=None, tb=None, serial=None):
        """gameplay::setup() + load_data() + _srand (gameplay.hpp:1231-1277, 1741-1925)."""
        ids = None if env_ids is None else np.ascontiguousarray(env_ids, dtype=np.int32)
        n = self.n_envs if ids is None else len(ids)
        tbv = None if tb is None else np.ascontiguousarray(tb, dtype=np.int64)
        sv = None if serial is None else np.ascontiguousarray(serial, dtype=np.int64)
        if tbv is not None:
            assert len(tbv) == n and len(sv) == n
        self._chk(lib().sf_reset(self._h, None if ids is None else ids.ctypes.data, n,
                                 None if tbv is None else tbv.ctypes.data, None if sv is None else sv.ctypes.data,
                                 self._stream()))

    def _act_ptr(self, actions):
        assert actions.is_cuda and actions.dtype == torch.uint8 and actions.is_contiguous()
        assert actions.numel() == self.n_envs * self.n_agents
        return C.c_void_p(actions.data_ptr())

    def step(self, actions):
        """One env-step of every arena (the loop body of gameplay::play, gameplay.hpp:1443-1472).
        ``actions``: uint8 device tensor [n_envs, n_agents] of command symbols."""
        self._chk(lib().sf_step(self._h, self._act_ptr(actions), self._stream()))
        self.step_count += 1

    def step_list(self, actions, env_ids, count=None):
        """sf_step_list: step the arenas of a device list and leave every other arena untouched.
        ``env_ids`` is an int32 CUDA tensor [n_max] and ``actions`` a uint8 CUDA tensor [n_max, n_agents] whose row i
        holds the commands of arena env_ids[i] (the row order of ``observe(env_ids=)``).  With ``count`` (an int32
        CUDA tensor [1], e.g. from ``list_finished``) only the first min(count, n_max) entries are live.  An id
        outside [0, n_envs) is skipped; a repeated id is stepped once, with the row of its first entry.  A listed
        arena ends as ``step`` with its row would leave it; the statistics count the stepped arenas only.  No host
        synchronisation; ``step_count`` is not advanced (the arenas no longer share one step number)."""
        assert env_ids.is_cuda and env_ids.dtype == torch.int32 and env_ids.is_contiguous() and env_ids.dim() == 1
        n_max = env_ids.numel()
        assert actions.is_cuda and actions.dtype == torch.uint8 and actions.is_contiguous()
        assert actions.numel() == n_max * self.n_agents
        if count is not None:
            assert count.is_cuda and count.dtype == torch.int32 and count.numel() == 1
        self._chk(lib().sf_step_list(self._h, C.c_void_p(actions.data_ptr()), C.c_void_p(env_ids.data_ptr()),
                                     None if count is None else C.c_void_p(count.data_ptr()), n_max, self._stream()))

    def step_a(self):
        self._chk(lib().sf_step_a(self._h, self._stream()))

    def step_b(self, actions):
        self._chk(lib().sf_step_b(self._h, self._act_ptr(actions), self._stream()))
        self.step_count += 1

    def step_host(self, actions_host, out_host):
        """The same step through HOST buffers: numpy uint8 [n_envs, n_agents] in, structured
        ``STEP_OUT_DTYPE`` [n_envs] out; copies both ways and synchronises."""
        assert actions_host.dtype == np.uint8 and actions_host.size == self.n_envs * self.n_agents
        assert out_host.dtype == sfcfg.STEP_OUT_DTYPE and out_host.size == self.n_envs
        self._chk(lib().sf_step_host(self._h, actions_host.ctypes.data, out_host.ctypes.data, self._stream()))
        self.step_count += 1

    def synth_actions(self, t, table=sfcfg.ACTIONS9, out=None):
        """Fill a device action buffer with the synthetic stream of include/sf_synth.h."""
        out = self._synth if out is None else out
        self._chk(lib().sf_synth_actions(self._h, self._act_ptr(out), int(t), bytes(table), len(table),
                                         self._stream()))
        return out

    # ------------------------------------------------------------------ observation / readback
    def observe(self, agent_mask=1, phase=sfcfg.OBS_P1, out=None, channels_last=False, env_ids=None, count=None,
                dtype=torch.float32):
        """gameplay::bot() up to Agent::predict (bots/bot-0.5/Custom.hpp:137-158): fp32 device
        tensor [n_envs, n_selected, 32, 31, 31].

        ``dtype=torch.float16`` or ``torch.bfloat16`` (SF_OBS_F16 / SF_OBS_BF16) writes half the bytes: every
        element equals ``.to(dtype)`` of the fp32 observation (round to nearest even), written by the
        observation kernel itself.  ``out`` must then have that dtype.

        ``channels_last=True`` returns a tensor of the same shape and values whose MEMORY is
        [n_envs, n_selected, 31, 31, 32] (SF_OBS_NHWC): ``.flatten(0, 1)`` of it is a channels-last batch that
        the policy's first convolution reads without a transpose.  ``out`` is always the plain buffer in memory
        order.

        ``env_ids`` (an int32 CUDA tensor [n_max], sf_observe_list) observes those arenas instead: the result has
        n_max rows, row i is arena env_ids[i] (duplicates allowed, an id outside [0, n_envs) gives a zero row).
        With ``count`` (an int32 CUDA tensor [1], e.g. from ``list_finished``) only the first min(count, n_max)
        rows are written, with no host synchronisation; rows at and beyond ``count`` are whatever ``out`` held
        (uninitialised memory when ``out`` is None)."""
        assert dtype in _OBS_FORMAT, "observations are float32, float16 or bfloat16"
        nsel = bin(agent_mask).count("1")
        W, CH = sfcfg.OBS_WIN, sfcfg.OBS_CH
        rows = self.n_envs
        if env_ids is not None:
            assert env_ids.is_cuda and env_ids.dtype == torch.int32 and env_ids.is_contiguous() and env_ids.dim() == 1
            rows = env_ids.numel()
            if count is not None:
                assert count.is_cuda and count.dtype == torch.int32 and count.numel() == 1
        else:
            assert count is None, "count goes with env_ids"
        if out is None:
            out = torch.empty((rows, nsel, W, W, CH) if channels_last else (rows, nsel, CH, W, W),
                              dtype=dtype, device=self.device)
        assert out.is_cuda and out.dtype == dtype and out.is_contiguous()
        assert out.numel() == rows * nsel * sfcfg.OBS_LEN
        ph = phase | (sfcfg.OBS_NHWC if channels_last else 0) | _OBS_FORMAT[dtype]
        if env_ids is None:
            self._chk(lib().sf_observe(self._h, C.c_void_p(out.data_ptr()), ph, agent_mask, self._stream()))
        else:
            self._chk(lib().sf_observe_list(self._h, C.c_void_p(out.data_ptr()), ph, agent_mask,
                                            C.c_void_p(env_ids.data_ptr()),
                                            None if count is None else C.c_void_p(count.data_ptr()), rows,
                                            self._stream()))
        if channels_last:
            return out.view(rows, nsel, W, W, CH).permute(0, 1, 4, 2, 3)
        return out

    def action_mask(self, env_ids=None, count=None, out=None, table=None):
        """sf_action_mask: which commands would change each driven human's arena now (include/strikeforce_b200.h,
        DESIGN.md section 7f).  An int32 CUDA tensor [rows, n_agents] of mask words: bit j stands for
        ``config.COMMANDS[j]`` (bit 31 is never set); a slot whose human the caller does not drive, or an arena that
        has ended, gets 0, and every other slot has the bit of '+'.

        ``env_ids`` / ``count`` follow ``observe(env_ids=, count=)``: row i is arena env_ids[i], an id outside
        [0, n_envs) gives a zero row, rows at and beyond ``count`` are whatever ``out`` held.  With ``table`` (bytes,
        e.g. ``config.ACTIONS9``) the result is instead a bool CUDA tensor [rows, n_agents, len(table)] whose
        [..., j] is the bit of table[j], computed on the device.  No host synchronisation either way."""
        rows = self.n_envs
        ids = cnt = None
        if env_ids is not None:
            ids = self._device_list(env_ids, "env_ids")
            rows = env_ids.numel()
            cnt = self._device_count(count)
        else:
            assert count is None, "count goes with env_ids"
        if out is None:
            out = torch.empty((rows, self.n_agents), dtype=torch.int32, device=self.device)
        assert out.is_cuda and out.dtype == torch.int32 and out.is_contiguous() and out.numel() == rows * self.n_agents
        self._chk(lib().sf_action_mask(self._h, C.c_void_p(out.data_ptr()), ids, cnt, rows, self._stream()))
        if table is None:
            return out
        table = bytes(table)
        bits = self._mask_bits.get(table)
        if bits is None:  # one copy per table, so that a captured graph holds no host-to-device copy
            bits = torch.tensor([sfcfg.COMMANDS.index(c) for c in table], dtype=torch.int32, device=self.device)
            self._mask_bits[table] = bits
        return ((out.unsqueeze(-1) >> bits) & 1).bool()

    # ------------------------------------------------------------------ finished arenas (final observations)
    def list_finished(self, ids=None, count=None):
        """sf_list_finished: ``(ids, count)``, device tensors int32 [n_envs] and int32 [1]: the ascending ids of
        the arenas whose episode has ended and that have not been reset since are ids[:count].  No host
        synchronisation; pass ``ids`` / ``count`` to reuse buffers (e.g. inside a CUDA graph)."""
        if ids is None:
            ids = torch.empty(self.n_envs, dtype=torch.int32, device=self.device)
        if count is None:
            count = torch.empty(1, dtype=torch.int32, device=self.device)
        assert ids.is_cuda and ids.dtype == torch.int32 and ids.is_contiguous() and ids.numel() == self.n_envs
        assert count.is_cuda and count.dtype == torch.int32 and count.numel() == 1
        self._chk(lib().sf_list_finished(self._h, C.c_void_p(ids.data_ptr()), C.c_void_p(count.data_ptr()),
                                         self._stream()))
        return ids, count

    def reset_finished(self):
        """sf_reset_finished: reset on the device every arena ``list_finished`` would list, as auto-reset would
        have at the end of the step that ended its episode.  With ``auto_reset=False`` and this call after every
        step, a run is the same as with auto-reset, but the terminal states can be observed in between (the
        "final observation" of a truncated episode).  No host synchronisation."""
        self._chk(lib().sf_reset_finished(self._h, self._stream()))

    def _get(self, field, shape, dtype):
        out = torch.empty(shape, dtype=dtype, device=self.device)
        self._chk(lib().sf_get(self._h, field, C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def step_out(self):
        """int32 [n_envs, 8]: status d_kills d_teams_kills d_loot d_hp d_damage d_effect episode_steps."""
        return self._get(sfcfg.FIELD_STEP_OUT, (self.n_envs, 8), torch.int32)

    def agent_out(self):
        """Per-agent step outputs (sf_get(SF_FIELD_AGENT_OUT), DESIGN.md section 7g): int32 CUDA tensor
        [n_envs, n_agents, 5], the fields ``config.AGENT_OUT_FIELDS`` (flags d_hp d_damage d_effect d_kills) of what
        the last step of each arena did to the human each column of the action row drives.  flags has
        ``config.AGENT_DRIVEN`` for a slot that was controllable when the step started (``action_mask() != 0``
        then) and ``config.AGENT_DIED`` when that human was gone at its end, before any auto-reset; a slot that was
        not driven is all zeros.  After ``step_list``, index it with the list's ids: unlisted arenas keep the rows
        of their own last step.  Needs ``agent_out=True`` at construction; no host synchronisation."""
        return self._get(sfcfg.FIELD_AGENT_OUT, (self.n_envs, self.n_agents, len(sfcfg.AGENT_OUT_FIELDS)), torch.int32)

    def match_logs(self, env_ids=None, count=None, out=None):
        """Match-log tapes (sf_log_list, DESIGN.md section 7h): a uint8 CUDA tensor [rows, sf_log_row_bytes], each
        row a ``config.LOG_HEAD`` (flags, status, level, episode, steps, n_symbols, tb, serial, global_id) and the
        tape's command symbols in the order of the reference's .sf_sample file; ``replay.write_device_log`` turns a
        row into a file.  ``env_ids`` / ``count`` follow ``action_mask``: row i is arena env_ids[i], an id outside
        [0, n_envs) gives an all-zero row, rows at and beyond ``count`` are whatever ``out`` held.  Needs
        ``match_log`` at construction; no host synchronisation."""
        row_bytes = lib().sf_log_row_bytes(self._h)
        rows, ids, cnt = self.n_envs, None, None
        if env_ids is not None:
            ids = self._device_list(env_ids, "env_ids")
            rows = env_ids.numel()
            cnt = self._device_count(count)
        else:
            assert count is None, "count goes with env_ids"
        if out is None:
            out = torch.empty((rows, row_bytes), dtype=torch.uint8, device=self.device)
        assert out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous() and out.numel() == rows * row_bytes
        self._chk(lib().sf_log_list(self._h, C.c_void_p(out.data_ptr()), ids, cnt, rows, self._stream()))
        return out

    def replay_load(self, rows, env_ids, count=None, status=None):
        """Load replay tapes (sf_replay_load, DESIGN.md section 7i): ``rows`` a uint8 CUDA tensor [n, row_bytes]
        in the layout ``match_logs()`` exports (``replay.tape_rows`` builds them from .sf_sample logs), ``env_ids``
        an int32 CUDA tensor [n]; row i resets arena env_ids[i] to the head's seeds, level and episode and arms its
        tape, and every later step deals the recorded commands from it in place of the action rows.  ``count`` (int32
        CUDA scalar) limits the live entries; an id outside [0, n_envs) is skipped, a repeated id loads from its
        lowest entry.  Returns the int32 CUDA ``status`` tensor, the number of refused entries (nothing is loaded
        unless it is 0), without reading it: no host synchronisation.  Needs ``replay`` at construction."""
        row_bytes = lib().sf_replay_row_bytes(self._h)
        n = env_ids.numel()
        assert rows.is_cuda and rows.dtype == torch.uint8 and rows.is_contiguous() and rows.numel() == n * row_bytes, \
            "rows: a uint8 CUDA tensor [n, sf_replay_row_bytes]"
        ids = self._device_list(env_ids, "env_ids")
        if status is None:
            status = torch.empty((), dtype=torch.int32, device=self.device)
        assert status.is_cuda and status.dtype == torch.int32 and status.numel() == 1
        self._chk(lib().sf_replay_load(self._h, C.c_void_p(rows.data_ptr()), ids, self._device_count(count), n,
                                       C.c_void_p(status.data_ptr()), self._stream()))
        return status

    def replay_state(self):
        """int32 CUDA tensor [n_envs, 5]: the ``config.REPLAY_STATE`` fields (flags cursor n_symbols steps status) of
        every arena's replay (sf_get(SF_FIELD_REPLAY)); no host synchronisation"""
        return self._get(sfcfg.FIELD_REPLAY, (self.n_envs, 5), torch.int32)

    def replay_dealt(self):
        """uint8 CUDA tensor [n_envs, n_agents]: the symbol each human slot took from its arena's tape in the arena's
        last step, as delivered to obey, 0 where none (sf_get(SF_FIELD_REPLAY_DEALT)) -- the action labels of a
        replayed step; no host synchronisation"""
        return self._get(sfcfg.FIELD_REPLAY_DEALT, (self.n_envs, self.n_agents), torch.uint8)

    def state_hash(self):
        return self._get(sfcfg.FIELD_STATE_HASH, (self.n_envs,), torch.int64)

    def counters(self):
        """int32 [n_envs, 8]: frame kills teams_kills loot chest steps status hp."""
        return self._get(sfcfg.FIELD_COUNTERS, (self.n_envs, 8), torch.int32)

    def population(self):
        """int32 [n_envs, 6]: humans zombies bullets chests built portals."""
        return self._get(sfcfg.FIELD_POPULATION, (self.n_envs, 6), torch.int32)

    def stats_tensor(self):
        """int64 [16] device-reduced running statistics (see config.STAT_NAMES)."""
        return self._get(sfcfg.FIELD_STATS, (16,), torch.int64)

    def stats(self):
        return dict(zip(sfcfg.STAT_NAMES, self.stats_tensor().cpu().tolist()))

    def export_env(self, env):
        """Canonical record (include/sf_canon.h) of one arena as a numpy int32 array."""
        buf = np.empty(1 << 18, dtype=np.int32)
        n = C.c_int64(buf.size)
        self._chk(lib().sf_export_env(self._h, env, buf.ctypes.data, C.byref(n)))
        return buf[:n.value].copy()

    # ------------------------------------------------------------------ arena records (sf_save / sf_load)
    @property
    def snapshot_bytes(self):
        """bytes of one arena record of this handle (include/strikeforce_b200.h, sf_snapshot_bytes)"""
        return int(lib().sf_snapshot_bytes(self._h))

    @staticmethod
    def _ids(ids):
        return None if ids is None else np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)

    @staticmethod
    def _device_list(t, what):
        assert t.is_cuda and t.dtype == torch.int32 and t.is_contiguous() and t.dim() == 1, \
            "%s: an int32 CUDA tensor [n_max]" % what
        return C.c_void_p(t.data_ptr())

    @staticmethod
    def _device_count(count):
        if count is None:
            return None
        assert count.is_cuda and count.dtype == torch.int32 and count.numel() == 1
        return C.c_void_p(count.data_ptr())

    def _record_buffer(self, out, n):
        if out is None:
            out = torch.empty((n, self.snapshot_bytes), dtype=torch.uint8, device=self.device)
        assert out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous()
        assert out.numel() == n * self.snapshot_bytes
        return out

    def save(self, env_ids=None, out=None, count=None):
        """Records of arenas ``env_ids`` (default: all, in order) as a uint8 device tensor
        [n, snapshot_bytes].  A checkpoint on disk is ``save().cpu().numpy()``.

        ``env_ids`` as an int32 CUDA tensor [n_max] (sf_save_list) saves a device list with no host
        synchronisation: row i is the record of arena env_ids[i] (duplicates allowed, an id outside [0, n_envs)
        gives an all-zero row that no load accepts).  With ``count`` (an int32 CUDA tensor [1]) only the first
        min(count, n_max) rows are written; the others are whatever ``out`` held."""
        if isinstance(env_ids, torch.Tensor) and env_ids.is_cuda:
            ids = self._device_list(env_ids, "env_ids")
            out = self._record_buffer(out, env_ids.numel())
            self._chk(lib().sf_save_list(self._h, C.c_void_p(out.data_ptr()), ids, self._device_count(count),
                                         env_ids.numel(), self._stream()))
            return out
        assert count is None, "count goes with a device env_ids"
        ids = self._ids(env_ids)
        n = self.n_envs if ids is None else len(ids)
        out = self._record_buffer(out, n)
        self._chk(lib().sf_save(self._h, None if ids is None else ids.ctypes.data, n, C.c_void_p(out.data_ptr()),
                                self._stream()))
        return out

    def load(self, records, env_ids=None, rows=None, count=None, status=None):
        """Overwrite arenas ``env_ids`` (default: all, in order; distinct) with the records ``records[rows[i]]``
        (default: row i).  ``records`` is a uint8 tensor [n_records, snapshot_bytes] (a host array or tensor is
        copied to the device first).  Raises (and changes no arena) when a record is not of this configuration.

        ``env_ids`` as an int32 CUDA tensor [n_max] (sf_load_list) loads a device list with no host
        synchronisation; ``records`` must then be a CUDA tensor and ``rows`` None or an int32 CUDA tensor [n_max].
        Only the first min(count, n_max) entries are live (``count``: an int32 CUDA tensor [1], None = all).  An id
        outside [0, n_envs) is skipped; a repeated id is loaded once, from its first entry.  All or nothing, decided
        on the device: the int32 CUDA tensor [1] returned (``status``, when given) holds the number of refused
        entries (a row outside the records, or a record of another configuration), and no arena changed unless it
        is 0.  It is not read back.

        Broadcast (one root into many slots): ``root = save(root_id)`` once, then ``load(root, slots,
        rows=zeros)``, with ``zeros`` an int32 CUDA tensor of zeros: every slot reads the same record, which stays
        in L2, instead of K copies of it."""
        if isinstance(env_ids, torch.Tensor) and env_ids.is_cuda:
            ids = self._device_list(env_ids, "env_ids")
            n_max = env_ids.numel()
            assert isinstance(records, torch.Tensor) and records.is_cuda and records.dtype == torch.uint8
            assert records.is_contiguous() and records.numel() % self.snapshot_bytes == 0
            rws = None if rows is None else self._device_list(rows, "rows")
            if rows is not None:
                assert rows.numel() == n_max
            if status is None:
                status = torch.empty(1, dtype=torch.int32, device=self.device)
            assert status.is_cuda and status.dtype == torch.int32 and status.numel() == 1
            self._chk(lib().sf_load_list(self._h, C.c_void_p(records.data_ptr()), records.numel() // self.snapshot_bytes,
                                         rws, ids, self._device_count(count), n_max, C.c_void_p(status.data_ptr()),
                                         self._stream()))
            return status
        assert count is None and status is None, "count and status go with a device env_ids"
        records = torch.as_tensor(records)
        if not records.is_cuda:
            records = records.to(self.device)
        records = records.contiguous().view(-1, self.snapshot_bytes)
        assert records.dtype == torch.uint8
        ids, rws = self._ids(env_ids), self._ids(rows)
        n = self.n_envs if ids is None else len(ids)
        if rws is not None:
            assert len(rws) == n
        self._chk(lib().sf_load(self._h, None if ids is None else ids.ctypes.data, n, C.c_void_p(records.data_ptr()),
                                records.shape[0], None if rws is None else rws.ctypes.data, self._stream()))

    def clone(self, src_ids, dst_ids, count=None, scratch=None, status=None):
        """Arena dst_ids[i] becomes a copy of arena src_ids[i]: one save of the distinct sources, one load.
        A copy under another global id goes on with the source's episode and then follows its own seeds.

        With int32 CUDA tensors [n_max] for both lists: ``save(src_ids, out=scratch, count=count)`` and then
        ``load(scratch, dst_ids, count=count, status=status)``, with no host synchronisation (a CUDA graph can
        capture it).  ``scratch`` is a uint8 CUDA tensor [n_max, snapshot_bytes] (allocated when None).  Returns
        the status tensor of the load: 0 when every listed destination was loaded; an out-of-range source gives a
        zero record, which refuses the whole clone if a destination in range takes it."""
        if isinstance(src_ids, torch.Tensor) and src_ids.is_cuda:
            assert isinstance(dst_ids, torch.Tensor) and dst_ids.is_cuda and dst_ids.numel() == src_ids.numel()
            scratch = self.save(src_ids, out=scratch, count=count)
            return self.load(scratch, dst_ids, count=count, status=status)
        assert count is None and scratch is None and status is None, "count, scratch and status go with device lists"
        src = self._ids(src_ids)
        uniq, rows = np.unique(src, return_inverse=True)
        self.load(self.save(uniq), dst_ids, rows=rows)

    def rng_stream(self, tb, serial, n_draws):
        """Random::_srand + n _rand() draws per stream on the device (random.hpp:54-76)."""
        tb = np.ascontiguousarray(tb, dtype=np.int64)
        serial = np.ascontiguousarray(serial, dtype=np.int64)
        out = np.empty((n_draws, len(tb)), dtype=np.int32)
        self._chk(lib().sf_rng_stream(self._h, tb.ctypes.data, serial.ctypes.data, len(tb), n_draws, out.ctypes.data))
        return out

    @property
    def launches(self):
        return int(lib().sf_launch_count(self._h))

    @property
    def device_bytes(self):
        return int(lib().sf_device_bytes(self._h))
