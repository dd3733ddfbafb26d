"""ctypes binding of tests/hostcheck/libsnapcheck.so: the host-check build (hostcheck.cpp) plus sf_save /
sf_load of one arena (snapcheck.cpp, csrc/sf_snapshot.cuh).  Debugging aid for the test-suite only."""
import ctypes as C
import os
import subprocess

import numpy as np

import hostcheck
from hostcheck import EXTRA, HERE, ROOT

# the entry points of hostcheck.cpp, bound here exactly as hostcheck.lib() binds them
_HC_NAMES = ("hc_create", "hc_destroy", "hc_reset", "hc_step", "hc_dump", "hc_hash", "hc_step_out", "hc_status",
             "hc_misc", "hc_stats", "hc_observe", "hc_n_agents")
_libs = {}


def lib_path(extra=EXTRA):
    return hostcheck.lib_path(extra).replace("libhostcheck", "libsnapcheck")


def build(force=False, extra=EXTRA):
    srcs = [os.path.join(HERE, f) for f in ("snapcheck.cpp", "hostcheck.cpp")] + [
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
        hc = hostcheck.lib(extra)
        for name in _HC_NAMES:
            f, g = getattr(L, name), getattr(hc, name)
            f.argtypes, f.restype = g.argtypes, g.restype
        L.hc_snapshot_bytes.argtypes = [C.c_void_p]
        L.hc_snapshot_bytes.restype = C.c_long
        L.hc_save.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.hc_load.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        _libs[extra] = L
    return _libs[extra]


class SnapSim(hostcheck.HostSim):
    """HostSim with arena records: save(env) / load(env, rec) as sf_save / sf_load do them for one arena"""

    def __init__(self, cfg, extra=EXTRA):
        self._cfg = cfg
        self._lib = lib(extra)
        self._h = self._lib.hc_create(C.byref(cfg))
        if not self._h:
            raise RuntimeError("hc_create failed")
        self.n_envs = cfg.n_envs
        self.n_agents = self._lib.hc_n_agents(self._h)

    @property
    def snapshot_bytes(self):
        return int(self._lib.hc_snapshot_bytes(self._h))

    def save(self, env):
        """the record of arena env (sf_save of the device library), uint8 [snapshot_bytes]"""
        rec = np.empty(self.snapshot_bytes, dtype=np.uint8)
        self._lib.hc_save(self._h, env, rec.ctypes.data)
        return rec

    def load(self, env, rec):
        """sf_load of one record into arena env; False (nothing changed) when the record is not of this configuration"""
        rec = np.ascontiguousarray(rec, dtype=np.uint8)
        assert rec.size == self.snapshot_bytes
        return self._lib.hc_load(self._h, env, rec.ctypes.data) == 0
