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


class BatchedArena:
    def __init__(self, n_envs, mode="Solo", level=1, level_max=None, squad_agents=False, auto_reset=True,
                 max_steps=0, env_id_base=0, player="account1", caps=None, arena=None, device=None, teams=None, sheets=None,
                 ind=0):
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
    def observe(self, agent_mask=1, phase=sfcfg.OBS_P1, out=None, channels_last=False, env_ids=None, count=None):
        """gameplay::bot() up to Agent::predict (bots/bot-0.5/Custom.hpp:137-158): fp32 device
        tensor [n_envs, n_selected, 32, 31, 31].

        ``channels_last=True`` returns a tensor of the same shape and values whose MEMORY is
        [n_envs, n_selected, 31, 31, 32] (SF_OBS_NHWC): ``.flatten(0, 1)`` of it is a channels-last batch that
        the policy's first convolution reads without a transpose.  ``out`` is always the plain buffer in memory
        order.

        ``env_ids`` (an int32 CUDA tensor [n_max], sf_observe_list) observes those arenas instead: the result has
        n_max rows, row i is arena env_ids[i] (duplicates allowed, an id outside [0, n_envs) gives a zero row).
        With ``count`` (an int32 CUDA tensor [1], e.g. from ``list_finished``) only the first min(count, n_max)
        rows are written, with no host synchronisation; rows at and beyond ``count`` are whatever ``out`` held
        (uninitialised memory when ``out`` is None)."""
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
                              dtype=torch.float32, device=self.device)
        assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous()
        assert out.numel() == rows * nsel * sfcfg.OBS_LEN
        ph = phase | (sfcfg.OBS_NHWC if channels_last else 0)
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

    def save(self, env_ids=None, out=None):
        """Records of arenas ``env_ids`` (default: all, in order) as a uint8 device tensor
        [n, snapshot_bytes].  A checkpoint on disk is ``save().cpu().numpy()``."""
        ids = self._ids(env_ids)
        n = self.n_envs if ids is None else len(ids)
        if out is None:
            out = torch.empty((n, self.snapshot_bytes), dtype=torch.uint8, device=self.device)
        assert out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous()
        assert out.numel() == n * self.snapshot_bytes
        self._chk(lib().sf_save(self._h, None if ids is None else ids.ctypes.data, n, C.c_void_p(out.data_ptr()),
                                self._stream()))
        return out

    def load(self, records, env_ids=None, rows=None):
        """Overwrite arenas ``env_ids`` (default: all, in order; distinct) with the records ``records[rows[i]]``
        (default: row i).  ``records`` is a uint8 tensor [n_records, snapshot_bytes] (a host array or tensor is
        copied to the device first).  Raises (and changes no arena) when a record is not of this configuration."""
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

    def clone(self, src_ids, dst_ids):
        """Arena dst_ids[i] becomes a copy of arena src_ids[i]: one save of the distinct sources, one load.
        A copy under another global id goes on with the source's episode and then follows its own seeds."""
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
