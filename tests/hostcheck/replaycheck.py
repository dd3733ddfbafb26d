"""ctypes binding of tests/hostcheck/libreplaycheck.so: the host-check build with match logs, arena records,
finished-arena calls, sf_step_list, the record lists, sf_action_mask and the per-agent step outputs (logcheck.cpp)
plus replay (replaycheck.cpp).  Debugging aid for the test-suite only."""
import ctypes as C
import os
import subprocess

import numpy as np

import hostcheck
import logcheck
from hostcheck import EXTRA, HERE, ROOT

_libs = {}


def lib_path(extra=EXTRA):
    return hostcheck.lib_path(extra).replace("libhostcheck", "libreplaycheck")


def build(force=False, extra=EXTRA):
    srcs = [os.path.join(HERE, f) for f in ("replaycheck.cpp", "logcheck.cpp", "agentcheck.cpp", "maskcheck.cpp",
                                            "reclistcheck.cpp", "listcheck.cpp", "finishcheck.cpp", "snapcheck.cpp",
                                            "hostcheck.cpp")] + [
        os.path.join(ROOT, "strikeforce_b200", "csrc", f)
        for f in ("sf_core.cuh", "sf_canon_dev.cuh", "sf_host_setup.h", "sf_state.h", "sf_obs.cuh", "sf_snapshot.cuh")] + [
        os.path.join(ROOT, "include", "strikeforce_b200.h")]
    path = lib_path(extra)
    if not force and os.path.exists(path) and all(os.path.getmtime(path) >= os.path.getmtime(s) for s in srcs):
        return
    subprocess.check_call([
        "g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"), "-I" + HERE,
        "-I" + os.path.join(ROOT, "strikeforce_b200", "csrc")] + list(extra) + ["-x", "c++", srcs[0], "-o", path])


def lib(extra=EXTRA):
    extra = tuple(extra)
    if extra not in _libs:
        build(extra=extra)
        L = C.CDLL(lib_path(extra))
        ll = logcheck.lib(extra)
        for name in dir(ll):  # the entry points of the files below, bound as logcheck binds them
            if name.startswith("hc_"):
                f, g = getattr(L, name), getattr(ll, name)
                f.argtypes, f.restype = g.argtypes, g.restype
        vp = C.c_void_p
        L.hc_enable_replay.argtypes = [vp, C.c_int]
        L.hc_enable_replay.restype = C.c_int
        L.hc_replay_row_bytes.argtypes = [vp]
        L.hc_replay_row_bytes.restype = C.c_int
        L.hc_disable_replay.argtypes = [vp]
        L.hc_step_replay.argtypes = [vp, C.c_char_p, C.c_int]
        L.hc_step_list_replay.argtypes = [vp, vp, C.c_int, vp]
        L.hc_replay_load.argtypes = [vp, vp, vp, C.c_int]
        L.hc_replay_load.restype = C.c_int
        L.hc_replay_state.argtypes = [vp, C.c_int, vp, vp]
        L.hc_replay_state.restype = C.c_int
        L.hc_reset_replay.argtypes = [vp, C.c_int, C.c_longlong, C.c_longlong]
        L.hc_load_replay.argtypes = [vp, C.c_int, vp]
        L.hc_load_replay.restype = C.c_int
        L.hc_load_list_replay.argtypes = [vp, vp, C.c_int, vp, vp, C.c_int]
        L.hc_load_list_replay.restype = C.c_int
        _libs[extra] = L
    return _libs[extra]


class ReplaySim(logcheck.LogSim):
    """LogSim with replay: after enable_replay(cap), step / step_list run sf_step_body<true> with every extra that is
    on as the EXTRAS kernels do, replay_load loads as sf_replay_load does, replay_state / replay_dealt read what
    sf_get(SF_FIELD_REPLAY / SF_FIELD_REPLAY_DEALT) reads, and reset / load / load_list disarm as the CUDA calls do"""

    def __init__(self, cfg, extra=EXTRA, agent_out=False, match_log=0, replay=0):
        self._cfg = cfg
        self._lib = lib(extra)
        self._h = self._lib.hc_create(C.byref(cfg))
        if not self._h:
            raise RuntimeError("hc_create failed")
        self.n_envs = cfg.n_envs
        self.n_agents = self._lib.hc_n_agents(self._h)
        self.agents = self.logging = self.replaying = False
        if agent_out:
            self.enable_agent_out()
        if match_log:
            assert self.enable_log(match_log)
        if replay:
            assert self.enable_replay(replay)

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.hc_disable_replay(self._h)  # keyed by the handle's address, like the tapes of the logs
        super().__del__()

    def enable_replay(self, cap):
        ok = self._lib.hc_enable_replay(self._h, cap) == 0
        self.replaying = self.replaying or ok
        return ok

    @property
    def replay_row_bytes(self):
        return self._lib.hc_replay_row_bytes(self._h)

    def step(self, actions, half=0):
        if not self.replaying:
            return super().step(actions, half)
        a = None if actions is None else bytes(actions)
        if a is not None:
            assert len(a) == self.n_envs * self.n_agents
        self._lib.hc_step_replay(self._h, a, half)

    def step_list(self, actions, ids):
        if not self.replaying:
            return super().step_list(actions, ids)
        ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        actions = np.ascontiguousarray(actions, dtype=np.uint8).reshape(len(ids), self.n_agents)
        self._lib.hc_step_list_replay(self._h, ids.ctypes.data, len(ids), actions.ctypes.data)

    def replay_load(self, rows, ids):
        """the number of refused owning entries (0: loaded)"""
        ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        rows = np.ascontiguousarray(rows, dtype=np.uint8).reshape(len(ids), self.replay_row_bytes)
        rc = self._lib.hc_replay_load(self._h, rows.ctypes.data, ids.ctypes.data, len(ids))
        assert rc >= 0, "replay is not enabled"
        return rc

    def replay_state(self, env):
        """(flags, cursor, n_symbols, steps, status)"""
        out, dealt = np.zeros(5, np.int32), np.zeros(self.n_agents, np.uint8)
        assert self._lib.hc_replay_state(self._h, env, out.ctypes.data, dealt.ctypes.data) == 0
        return tuple(int(x) for x in out)

    def replay_dealt(self, env):
        out, dealt = np.zeros(5, np.int32), np.zeros(self.n_agents, np.uint8)
        assert self._lib.hc_replay_state(self._h, env, out.ctypes.data, dealt.ctypes.data) == 0
        return dealt

    def reset(self, env, tb, serial):
        self._lib.hc_reset_replay(self._h, env, tb, serial)

    def load(self, env, rec):
        rec = np.ascontiguousarray(rec, dtype=np.uint8)
        assert rec.size == self.snapshot_bytes
        return self._lib.hc_load_replay(self._h, env, rec.ctypes.data) == 0

    def load_list(self, records, ids, rows=None, count=None):
        records = np.ascontiguousarray(records, dtype=np.uint8).reshape(-1, self.snapshot_bytes)
        ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        rws = None if rows is None else np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
        n = len(ids) if count is None else max(0, min(int(count), len(ids)))
        return self._lib.hc_load_list_replay(self._h, records.ctypes.data, len(records),
                                             None if rws is None else rws.ctypes.data, ids.ctypes.data, n)
