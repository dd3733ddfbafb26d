"""ctypes binding of tests/hostcheck/liblistcheck.so: the host-check build with arena records and finished-arena
calls (finishcheck.cpp) plus sf_step_list (listcheck.cpp).  Debugging aid for the test-suite only."""
import ctypes as C
import os
import subprocess

import numpy as np

import finishcheck
import hostcheck
import snapcheck
from hostcheck import EXTRA, HERE, ROOT

_libs = {}


def lib_path(extra=EXTRA):
    return hostcheck.lib_path(extra).replace("libhostcheck", "liblistcheck")


def build(force=False, extra=EXTRA):
    srcs = [os.path.join(HERE, f) for f in ("listcheck.cpp", "finishcheck.cpp", "snapcheck.cpp", "hostcheck.cpp")] + [
        os.path.join(ROOT, "strikeforce_b200", "csrc", f)
        for f in ("sf_core.cuh", "sf_canon_dev.cuh", "sf_host_setup.h", "sf_state.h", "sf_obs.cuh", "sf_snapshot.cuh")]
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
        fin = finishcheck.lib(extra)
        # the entry points of hostcheck.cpp, snapcheck.cpp and finishcheck.cpp, bound as their own modules bind them
        for name in snapcheck._HC_NAMES + finishcheck._SNAP_NAMES + ("hc_reset_finished", "hc_list_finished"):
            f, g = getattr(L, name), getattr(fin, name)
            f.argtypes, f.restype = g.argtypes, g.restype
        L.hc_step_list.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        _libs[extra] = L
    return _libs[extra]


class ListSim(finishcheck.FinishSim):
    """FinishSim with step_list(actions, ids) as sf_step_list does it"""

    def __init__(self, cfg, extra=EXTRA):
        self._cfg = cfg
        self._lib = lib(extra)
        self._h = self._lib.hc_create(C.byref(cfg))
        if not self._h:
            raise RuntimeError("hc_create failed")
        self.n_envs = cfg.n_envs
        self.n_agents = self._lib.hc_n_agents(self._h)

    def step_list(self, actions, ids):
        """sf_step_list: ids int32 [n], actions uint8 [n, n_agents], row i for entry i"""
        ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        actions = np.ascontiguousarray(actions, dtype=np.uint8).reshape(len(ids), self.n_agents)
        self._lib.hc_step_list(self._h, ids.ctypes.data, len(ids), actions.ctypes.data)
