"""ctypes binding of tests/hostcheck/libfinishcheck.so: the host-check build with arena records (snapcheck.cpp)
plus sf_reset_finished / sf_list_finished over all arenas (finishcheck.cpp).  Debugging aid for the test-suite
only."""
import ctypes as C
import os
import subprocess

import numpy as np

import hostcheck
import snapcheck
from hostcheck import EXTRA, HERE, ROOT

# the entry points of hostcheck.cpp and snapcheck.cpp, bound here exactly as their own modules bind them
_SNAP_NAMES = ("hc_snapshot_bytes", "hc_save", "hc_load")
_libs = {}


def lib_path(extra=EXTRA):
    return hostcheck.lib_path(extra).replace("libhostcheck", "libfinishcheck")


def build(force=False, extra=EXTRA):
    srcs = [os.path.join(HERE, f) for f in ("finishcheck.cpp", "snapcheck.cpp", "hostcheck.cpp")] + [
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
        snap = snapcheck.lib(extra)
        for name in snapcheck._HC_NAMES + _SNAP_NAMES:
            f, g = getattr(L, name), getattr(snap, name)
            f.argtypes, f.restype = g.argtypes, g.restype
        L.hc_reset_finished.argtypes = [C.c_void_p]
        L.hc_list_finished.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _libs[extra] = L
    return _libs[extra]


class FinishSim(snapcheck.SnapSim):
    """SnapSim with reset_finished() / list_finished() as sf_reset_finished / sf_list_finished do them"""

    def __init__(self, cfg, extra=EXTRA):
        self._cfg = cfg
        self._lib = lib(extra)
        self._h = self._lib.hc_create(C.byref(cfg))
        if not self._h:
            raise RuntimeError("hc_create failed")
        self.n_envs = cfg.n_envs
        self.n_agents = self._lib.hc_n_agents(self._h)

    def reset_finished(self):
        """sf_reset_finished: reset every arena whose episode has ended, as auto-reset would have"""
        self._lib.hc_reset_finished(self._h)

    def list_finished(self):
        """sf_list_finished: the ascending ids of the arenas whose episode has ended (numpy int32)"""
        ids = np.empty(self.n_envs, dtype=np.int32)
        n = np.zeros(1, dtype=np.int32)
        self._lib.hc_list_finished(self._h, ids.ctypes.data, n.ctypes.data)
        return ids[:int(n[0])].copy()
