"""ctypes wrapper of tests/emu/dyn_sampler.cpp: the per-env dynamics sampler of solo_env.cuh built for the host
(TEST HARNESS ONLY)."""
import ctypes as C
import os
import subprocess

import numpy as np

from solorl_b200.abi import SoloSimParams

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = os.path.join(_ROOT, "tests", "_build", "libsolo_dyn_sampler.so")
_lib = None


def build():
    srcs = [os.path.join(_HERE, "dyn_sampler.cpp")] + [
        os.path.join(_ROOT, "solorl_b200", "csrc", f) for f in ("solo_core.cuh", "solo_env.cuh", "solo_host_model.h")] + [
        os.path.join(_ROOT, "include", "solo_b200.h")]
    if (not os.path.exists(_LIB)) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in srcs):
        os.makedirs(os.path.dirname(_LIB), exist_ok=True)
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared",
                               "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", _LIB, srcs[0]])
    return _LIB


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.dyn_sample.argtypes = [C.POINTER(SoloSimParams), C.c_uint64, C.c_int64, C.c_int, C.c_uint32,
                                 C.POINTER(C.c_float)]
        _lib = L
    return _lib


def sample(params, seed, gid0, n, episode):
    """float32 [n,3] = (friction, base mass scale, motor strength) that a randomised handle draws at the reset
    starting episode ``episode`` (1 for the first reset) of the envs with global ids gid0 .. gid0+n-1."""
    out = np.zeros((n, 3), np.float32)
    rc = lib().dyn_sample(C.byref(params), int(seed) & (2 ** 64 - 1), int(gid0), int(n), int(episode),
                          out.ctypes.data_as(C.POINTER(C.c_float)))
    if rc != 0:
        raise ValueError(f"dyn_sample rejected the ranges (rc {rc})")
    return out
