"""ctypes binding of tests/hostcheck/libagentcheck.so: the host-check build with arena records, finished-arena calls,
sf_step_list, the record lists and sf_action_mask (maskcheck.cpp) plus the per-agent step outputs (agentcheck.cpp).
Debugging aid for the test-suite only."""
import ctypes as C
import os
import subprocess

import numpy as np

import finishcheck
import hostcheck
import maskcheck
import snapcheck
from hostcheck import EXTRA, HERE, ROOT

_libs = {}


def lib_path(extra=EXTRA):
    return hostcheck.lib_path(extra).replace("libhostcheck", "libagentcheck")


def build(force=False, extra=EXTRA):
    srcs = [os.path.join(HERE, f) for f in ("agentcheck.cpp", "maskcheck.cpp", "reclistcheck.cpp", "listcheck.cpp",
                                            "finishcheck.cpp", "snapcheck.cpp", "hostcheck.cpp")] + [
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
        ml = maskcheck.lib(extra)
        # the entry points of the files below, bound as their own modules bind them
        for name in snapcheck._HC_NAMES + finishcheck._SNAP_NAMES + (
                "hc_reset_finished", "hc_list_finished", "hc_step_list", "hc_save_list", "hc_load_list",
                "hc_action_mask", "hc_action_mask_brute", "hc_commands"):
            f, g = getattr(L, name), getattr(ml, name)
            f.argtypes, f.restype = g.argtypes, g.restype
        L.hc_enable_agent_out.argtypes = [C.c_void_p]
        L.hc_disable_agent_out.argtypes = [C.c_void_p]
        L.hc_step_agents.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.hc_step_list_agents.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.hc_agent_out.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.hc_agent_out.restype = C.c_int
        _libs[extra] = L
    return _libs[extra]


class AgentSim(maskcheck.MaskSim):
    """MaskSim with agent outputs: after enable_agent_out(), step / step_list run sf_step_body<true> as the AGENTS
    kernels do, and agent_out() reads the rows as sf_get(SF_FIELD_AGENT_OUT) does"""

    def __init__(self, cfg, extra=EXTRA, agent_out=False):
        self._cfg = cfg
        self._lib = lib(extra)
        self._h = self._lib.hc_create(C.byref(cfg))
        if not self._h:
            raise RuntimeError("hc_create failed")
        self.n_envs = cfg.n_envs
        self.n_agents = self._lib.hc_n_agents(self._h)
        self.agents = False
        if agent_out:
            self.enable_agent_out()

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.hc_disable_agent_out(self._h)  # the rows are keyed by the handle's address
        super().__del__()

    def enable_agent_out(self):
        self._lib.hc_enable_agent_out(self._h)
        self.agents = True

    def step(self, actions, half=0):
        if not self.agents:
            return super().step(actions, half)
        a = None if actions is None else bytes(actions)
        if a is not None:
            assert len(a) == self.n_envs * self.n_agents
        self._lib.hc_step_agents(self._h, a, half)

    def step_list(self, actions, ids):
        if not self.agents:
            return super().step_list(actions, ids)
        ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        actions = np.ascontiguousarray(actions, dtype=np.uint8).reshape(len(ids), self.n_agents)
        self._lib.hc_step_list_agents(self._h, ids.ctypes.data, len(ids), actions.ctypes.data)

    def agent_out(self, env=None):
        """int32 [n_agents, 5] of arena env, or [n_envs, n_agents, 5] of every arena"""
        if env is None:
            return np.stack([self.agent_out(e) for e in range(self.n_envs)])
        out = np.zeros((self.n_agents, 5), dtype=np.int32)
        assert self._lib.hc_agent_out(self._h, env, out.ctypes.data) == 0, "agent outputs are not enabled"
        return out
