"""ctypes binding of tests/hostcheck/libreclistcheck.so: the host-check build with arena records, finished-arena calls
and sf_step_list (listcheck.cpp) plus sf_save_list / sf_load_list (reclistcheck.cpp).  Debugging aid for the
test-suite only."""
import ctypes as C
import os
import subprocess

import numpy as np

import finishcheck
import hostcheck
import listcheck
import snapcheck
from hostcheck import EXTRA, HERE, ROOT

_libs = {}


def lib_path(extra=EXTRA):
    return hostcheck.lib_path(extra).replace("libhostcheck", "libreclistcheck")


def build(force=False, extra=EXTRA):
    srcs = [os.path.join(HERE, f) for f in ("reclistcheck.cpp", "listcheck.cpp", "finishcheck.cpp", "snapcheck.cpp",
                                            "hostcheck.cpp")] + [
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
        lst = listcheck.lib(extra)
        # the entry points of the files below, bound as their own modules bind them
        for name in snapcheck._HC_NAMES + finishcheck._SNAP_NAMES + ("hc_reset_finished", "hc_list_finished",
                                                                      "hc_step_list"):
            f, g = getattr(L, name), getattr(lst, name)
            f.argtypes, f.restype = g.argtypes, g.restype
        L.hc_save_list.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.hc_load_list.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.hc_load_list.restype = C.c_int
        _libs[extra] = L
    return _libs[extra]


class RecListSim(listcheck.ListSim):
    """ListSim with save_list / load_list as sf_save_list / sf_load_list do them"""

    def __init__(self, cfg, extra=EXTRA):
        self._cfg = cfg
        self._lib = lib(extra)
        self._h = self._lib.hc_create(C.byref(cfg))
        if not self._h:
            raise RuntimeError("hc_create failed")
        self.n_envs = cfg.n_envs
        self.n_agents = self._lib.hc_n_agents(self._h)

    def save_list(self, ids, out=None, count=None):
        """sf_save_list: writes rows i < count (default: all) of out (uint8 [len(ids), snapshot_bytes]) and returns it"""
        ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        if out is None:
            out = np.zeros((len(ids), self.snapshot_bytes), dtype=np.uint8)
        assert out.dtype == np.uint8 and out.flags.c_contiguous and out.size == len(ids) * self.snapshot_bytes
        n = len(ids) if count is None else max(0, min(int(count), len(ids)))
        self._lib.hc_save_list(self._h, ids.ctypes.data, n, out.ctypes.data)
        return out

    def load_list(self, records, ids, rows=None, count=None):
        """sf_load_list: the number of refused owning entries (0: the listed arenas were loaded)"""
        records = np.ascontiguousarray(records, dtype=np.uint8).reshape(-1, self.snapshot_bytes)
        ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        rws = None if rows is None else np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
        n = len(ids) if count is None else max(0, min(int(count), len(ids)))
        return self._lib.hc_load_list(self._h, records.ctypes.data, len(records),
                                      None if rws is None else rws.ctypes.data, ids.ctypes.data, n)
