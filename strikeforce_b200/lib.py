"""ctypes binding of ``libstrikeforce_b200.so`` -- the C ABI of ``include/strikeforce_b200.h``.

There is no Python or CPU implementation behind these calls: if the CUDA library is missing
or no CUDA device is usable every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

from . import config as sfcfg

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SF_LIB_PATH") or os.path.join(_HERE, "libstrikeforce_b200%s.so" % sfcfg.GEOMETRY_TAG)
BUILD_SCRIPT = os.path.join(_HERE, "csrc", "build.sh")

EXPORTS = [
    "sf_abi_version", "sf_last_error", "sf_create", "sf_destroy", "sf_reset", "sf_step", "sf_step_a", "sf_step_b",
    "sf_step_host", "sf_step_list", "sf_synth_actions", "sf_observe", "sf_list_finished", "sf_reset_finished", "sf_observe_list",
    "sf_get", "sf_export_env", "sf_snapshot_bytes", "sf_save", "sf_load", "sf_save_list", "sf_load_list",
    "sf_rng_stream", "sf_agents_per_env", "sf_num_envs", "sf_launch_count", "sf_device_bytes", "sf_action_mask",
    "sf_enable_agent_out", "sf_enable_log", "sf_log_row_bytes", "sf_log_list", "sf_enable_replay", "sf_replay_row_bytes",
    "sf_replay_load",
]

_lib = None


class SfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("strikeforce_b200: %s (%d): %s" % (sfcfg.ERRORS.get(code, "error"), code, msg))
        self.code = code


def build(force=False):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(_HERE, "csrc", f) for f in os.listdir(os.path.join(_HERE, "csrc"))]
    srcs += [os.path.join(os.path.dirname(_HERE), "include", f)
             for f in ("strikeforce_b200.h", "sf_canon.h", "sf_synth.h")]
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs):
        return LIB_PATH
    subprocess.check_call(["bash", BUILD_SCRIPT])
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SfError(-2, "%s is missing: run strikeforce_b200.lib.build() (needs nvcc); "
                              "there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
        L.sf_abi_version.restype = i32
        L.sf_last_error.argtypes = [vp]
        L.sf_last_error.restype = C.c_char_p
        L.sf_create.argtypes = [C.POINTER(sfcfg.SfConfig), C.POINTER(vp)]
        L.sf_destroy.argtypes = [vp]
        L.sf_reset.argtypes = [vp, vp, i32, vp, vp, vp]
        L.sf_step.argtypes = [vp, vp, vp]
        L.sf_step_a.argtypes = [vp, vp]
        L.sf_step_b.argtypes = [vp, vp, vp]
        L.sf_step_host.argtypes = [vp, vp, vp, vp]
        L.sf_step_list.argtypes = [vp, vp, vp, vp, i32, vp]
        L.sf_synth_actions.argtypes = [vp, vp, u64, C.c_char_p, i32, vp]
        L.sf_observe.argtypes = [vp, vp, i32, C.c_uint32, vp]
        L.sf_list_finished.argtypes = [vp, vp, vp, vp]
        L.sf_reset_finished.argtypes = [vp, vp]
        L.sf_observe_list.argtypes = [vp, vp, i32, C.c_uint32, vp, vp, i32, vp]
        L.sf_get.argtypes = [vp, i32, vp, vp]
        L.sf_export_env.argtypes = [vp, i32, vp, C.POINTER(i64)]
        L.sf_snapshot_bytes.argtypes = [vp]
        L.sf_snapshot_bytes.restype = i64
        L.sf_save.argtypes = [vp, vp, i32, vp, vp]
        L.sf_load.argtypes = [vp, vp, i32, vp, i32, vp, vp]
        L.sf_save_list.argtypes = [vp, vp, vp, vp, i32, vp]
        L.sf_load_list.argtypes = [vp, vp, i32, vp, vp, vp, i32, vp, vp]
        L.sf_action_mask.argtypes = [vp, vp, vp, vp, i32, vp]
        L.sf_enable_agent_out.argtypes = [vp]
        L.sf_enable_log.argtypes = [vp, i32]
        L.sf_log_row_bytes.argtypes = [vp]
        L.sf_log_list.argtypes = [vp, vp, vp, vp, i32, vp]
        L.sf_enable_replay.argtypes = [vp, i32]
        L.sf_replay_row_bytes.argtypes = [vp]
        L.sf_replay_load.argtypes = [vp, vp, vp, vp, i32, vp, vp]
        L.sf_rng_stream.argtypes = [vp, vp, vp, i32, i32, vp]
        L.sf_agents_per_env.argtypes = [vp]
        L.sf_num_envs.argtypes = [vp]
        L.sf_launch_count.argtypes = [vp]
        L.sf_launch_count.restype = i64
        L.sf_device_bytes.argtypes = [vp]
        L.sf_device_bytes.restype = i64
        if L.sf_abi_version() != sfcfg.ABI_VERSION:
            raise SfError(-4, "ABI version mismatch between %s and the Python mirror" % LIB_PATH)
        _lib = L
    return _lib


def check(rc, handle=None):
    if rc != 0:
        msg = lib().sf_last_error(handle)
        raise SfError(rc, msg.decode() if msg else "")
