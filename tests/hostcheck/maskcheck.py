"""ctypes binding of tests/hostcheck/libmaskcheck.so: the host-check build with arena records, finished-arena calls,
sf_step_list and the record lists (reclistcheck.cpp) plus sf_action_mask (maskcheck.cpp).  Debugging aid for the
test-suite only."""
import ctypes as C
import os
import subprocess

import numpy as np

import finishcheck
import hostcheck
import reclistcheck
import snapcheck
from hostcheck import EXTRA, HERE, ROOT

_libs = {}


def lib_path(extra=EXTRA):
    return hostcheck.lib_path(extra).replace("libhostcheck", "libmaskcheck")


def build(force=False, extra=EXTRA):
    srcs = [os.path.join(HERE, f) for f in ("maskcheck.cpp", "reclistcheck.cpp", "listcheck.cpp", "finishcheck.cpp",
                                            "snapcheck.cpp", "hostcheck.cpp")] + [
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
        rl = reclistcheck.lib(extra)
        # the entry points of the files below, bound as their own modules bind them
        for name in snapcheck._HC_NAMES + finishcheck._SNAP_NAMES + ("hc_reset_finished", "hc_list_finished",
                                                                      "hc_step_list", "hc_save_list", "hc_load_list"):
            f, g = getattr(L, name), getattr(rl, name)
            f.argtypes, f.restype = g.argtypes, g.restype
        L.hc_action_mask.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.hc_action_mask_brute.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.hc_action_mask_brute.restype = C.c_int
        L.hc_commands.restype = C.c_char_p
        _libs[extra] = L
    return _libs[extra]


def commands(extra=EXTRA):
    """SF_COMMANDS as the header defines it"""
    return lib(extra).hc_commands()


class MaskSim(reclistcheck.RecListSim):
    """RecListSim with action_mask(env) as sf_action_mask computes it, and action_mask_brute(env) by the definition"""

    def __init__(self, cfg, extra=EXTRA):
        self._cfg = cfg
        self._lib = lib(extra)
        self._h = self._lib.hc_create(C.byref(cfg))
        if not self._h:
            raise RuntimeError("hc_create failed")
        self.n_envs = cfg.n_envs
        self.n_agents = self._lib.hc_n_agents(self._h)

    def action_mask(self, env):
        out = np.zeros(self.n_agents, dtype=np.uint32)
        self._lib.hc_action_mask(self._h, env, out.ctypes.data)
        return out

    def action_mask_brute(self, env):
        out = np.zeros(self.n_agents, dtype=np.uint32)
        assert self._lib.hc_action_mask_brute(self._h, env, out.ctypes.data) == 0, \
            "arena %d: a restored record differs from the one saved" % env
        return out

    def masks(self, brute=False):
        """uint32 [n_envs, n_agents]"""
        f = self.action_mask_brute if brute else self.action_mask
        return np.stack([f(e) for e in range(self.n_envs)])
