"""ctypes binding of tests/hostcheck/liblogcheck.so: the host-check build with arena records, finished-arena calls,
sf_step_list, the record lists, sf_action_mask and the per-agent step outputs (agentcheck.cpp) plus the match logs
(logcheck.cpp).  Debugging aid for the test-suite only."""
import ctypes as C
import os
import subprocess

import numpy as np

import agentcheck
import hostcheck
from hostcheck import EXTRA, HERE, ROOT

_libs = {}


def lib_path(extra=EXTRA):
    return hostcheck.lib_path(extra).replace("libhostcheck", "liblogcheck")


def build(force=False, extra=EXTRA):
    srcs = [os.path.join(HERE, f) for f in ("logcheck.cpp", "agentcheck.cpp", "maskcheck.cpp", "reclistcheck.cpp",
                                            "listcheck.cpp", "finishcheck.cpp", "snapcheck.cpp", "hostcheck.cpp")] + [
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
        al = agentcheck.lib(extra)
        for name in dir(al):  # the entry points of the files below, bound as agentcheck binds them
            if name.startswith("hc_"):
                f, g = getattr(L, name), getattr(al, name)
                f.argtypes, f.restype = g.argtypes, g.restype
        L.hc_enable_log.argtypes = [C.c_void_p, C.c_int]
        L.hc_enable_log.restype = C.c_int
        L.hc_log_row_bytes.argtypes = [C.c_void_p]
        L.hc_log_row_bytes.restype = C.c_int
        L.hc_disable_log.argtypes = [C.c_void_p]
        L.hc_step_log.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.hc_step_list_log.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.hc_log_list.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.hc_log_list.restype = C.c_int
        L.hc_load_log.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.hc_load_log.restype = C.c_int
        L.hc_load_list_log.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.hc_load_list_log.restype = C.c_int
        _libs[extra] = L
    return _libs[extra]


class LogSim(agentcheck.AgentSim):
    """AgentSim with match logs: after enable_log(cap), step / step_list run sf_step_body<true> with the tapes as
    the EXTRAS kernels do, logs() exports rows as sf_log_list does, and load / load_list clear SF_LOG_COMPLETE as
    sf_load / sf_load_list do"""

    def __init__(self, cfg, extra=EXTRA, agent_out=False, match_log=0):
        self._cfg = cfg
        self._lib = lib(extra)
        self._h = self._lib.hc_create(C.byref(cfg))
        if not self._h:
            raise RuntimeError("hc_create failed")
        self.n_envs = cfg.n_envs
        self.n_agents = self._lib.hc_n_agents(self._h)
        self.agents = self.logging = False
        if agent_out:
            self.enable_agent_out()
        if match_log:
            assert self.enable_log(match_log)

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.hc_disable_log(self._h)  # the tapes are keyed by the handle's address
        super().__del__()

    def enable_log(self, cap):
        ok = self._lib.hc_enable_log(self._h, cap) == 0
        self.logging = self.logging or ok
        return ok

    @property
    def row_bytes(self):
        return self._lib.hc_log_row_bytes(self._h)

    def step(self, actions, half=0):
        if not self.logging:
            return super().step(actions, half)
        a = None if actions is None else bytes(actions)
        if a is not None:
            assert len(a) == self.n_envs * self.n_agents
        self._lib.hc_step_log(self._h, a, half)

    def step_list(self, actions, ids):
        if not self.logging:
            return super().step_list(actions, ids)
        ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        actions = np.ascontiguousarray(actions, dtype=np.uint8).reshape(len(ids), self.n_agents)
        self._lib.hc_step_list_log(self._h, ids.ctypes.data, len(ids), actions.ctypes.data)

    def logs(self, ids=None):
        """uint8 [rows, row_bytes]: the tapes of arenas ids (default: all), as sf_log_list exports them"""
        n = self.n_envs if ids is None else len(ids)
        out = np.empty((n, self.row_bytes), dtype=np.uint8)
        idp = None
        if ids is not None:
            ids = np.ascontiguousarray(ids, dtype=np.int32)
            idp = ids.ctypes.data
        assert self._lib.hc_log_list(self._h, idp, n, out.ctypes.data) == 0, "match logs are not enabled"
        return out

    def load(self, env, rec):
        rec = np.ascontiguousarray(rec, dtype=np.uint8)
        assert rec.size == self.snapshot_bytes
        return self._lib.hc_load_log(self._h, env, rec.ctypes.data) == 0

    def load_list(self, records, ids, rows=None, count=None):
        records = np.ascontiguousarray(records, dtype=np.uint8).reshape(-1, self.snapshot_bytes)
        ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        rws = None if rows is None else np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
        n = len(ids) if count is None else max(0, min(int(count), len(ids)))
        return self._lib.hc_load_list_log(self._h, records.ctypes.data, len(records),
                                          None if rws is None else rws.ctypes.data, ids.ctypes.data, n)


def heads(rows):
    """the sf_log_head of every row (numpy structured array)"""
    from strikeforce_b200 import config as sfcfg
    return np.ascontiguousarray(rows[:, :sfcfg.LOG_HEAD.itemsize]).view(sfcfg.LOG_HEAD).reshape(-1)


def tape(row):
    from strikeforce_b200 import config as sfcfg
    n = int(heads(row[None])[0]["n_symbols"])
    return row[sfcfg.LOG_HEAD.itemsize:sfcfg.LOG_HEAD.itemsize + n].tobytes()
