"""ctypes binding of tests/hostcheck/libbtcheck.so: the host-check build with arena records (snapcheck.cpp) plus the
bullet-flag table of the tick, entry by entry (btcheck.cpp).  Debugging aid for the test-suite only."""
import ctypes as C
import os
import subprocess

import numpy as np

import hostcheck
import snapcheck
from hostcheck import EXTRA, HERE, ROOT

_SNAP_NAMES = ("hc_snapshot_bytes", "hc_save", "hc_load")
_libs = {}


def lib_path(extra=EXTRA):
    return hostcheck.lib_path(extra).replace("libhostcheck", "libbtcheck")


def build(force=False, extra=EXTRA):
    srcs = [os.path.join(HERE, f) for f in ("btcheck.cpp", "snapcheck.cpp", "hostcheck.cpp")] + [
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
        L.hc_bt_wipe.argtypes = [C.c_void_p, C.c_int]
        L.hc_bt_flag.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.hc_bt_flag.restype = C.c_uint
        L.hc_bt_flagged.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.hc_bt_count.argtypes = [C.c_void_p]
        L.hc_bt_count.restype = C.c_uint
        L.hc_bt_rebuild.argtypes = [C.c_void_p, C.c_int]
        L.hc_bt_owners.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.hc_bt_geometry.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_int)]
        _libs[extra] = L
    return _libs[extra]


def geometry(extra=EXTRA):
    """(buckets, SF_BT_FULL, number of cell ids) of the build"""
    full, cells = C.c_int(), C.c_int()
    n = lib(extra).hc_bt_geometry(C.byref(full), C.byref(cells))
    return n, full.value, cells.value


class BtSim(snapcheck.SnapSim):
    """SnapSim with the bullet-flag table of the tick exposed entry by entry"""

    def __init__(self, cfg, extra=EXTRA):
        self._cfg = cfg
        self._lib = lib(extra)
        self._h = self._lib.hc_create(C.byref(cfg))
        if not self._h:
            raise RuntimeError("hc_create failed")
        self.n_envs = cfg.n_envs
        self.n_agents = self._lib.hc_n_agents(self._h)

    def bt_wipe(self, env):
        self._lib.hc_bt_wipe(self._h, env)

    def bt_flag(self, env, cell):
        return self._lib.hc_bt_flag(self._h, env, cell)

    def bt_flagged(self, env, cell):
        return bool(self._lib.hc_bt_flagged(self._h, env, cell))

    def bt_count(self):
        return self._lib.hc_bt_count(self._h)

    def bt_rebuild(self, env):
        self._lib.hc_bt_rebuild(self._h, env)

    def bt_owners(self, env):
        """(cells, spilled) of the live bullets of arena env that own a flag, in slot order (numpy)"""
        cells, spilled = np.empty(128, dtype=np.int32), np.empty(128, dtype=np.int32)
        n = self._lib.hc_bt_owners(self._h, env, cells.ctypes.data, spilled.ctypes.data)
        return cells[:n].copy(), spilled[:n].astype(bool)
