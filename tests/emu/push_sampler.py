"""ctypes wrapper of tests/emu/push_sampler.cpp: the random push schedule of solo_env.cuh built for the host
(TEST HARNESS ONLY)."""
import ctypes as C
import os
import subprocess

import numpy as np

from solorl_b200.abi import SoloSimParams

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = os.path.join(_ROOT, "tests", "_build", "libsolo_push_sampler.so")
_lib = None


def build():
    srcs = [os.path.join(_HERE, "push_sampler.cpp")] + [
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
        L.push_sample.argtypes = [C.POINTER(SoloSimParams), C.c_uint64, C.c_int64, C.c_int, C.c_uint32, C.c_int32,
                                  C.c_int, C.POINTER(C.c_float)]
        _lib = L
    return _lib


def push_sample(params, seed, gid0, n, episode, t0, T):
    """float32 [n,T,3] = the push (fx, fy, 0) of control steps t0 .. t0+T-1 (steps completed in the episode) of
    episode ``episode`` of the envs with global ids gid0 .. gid0+n-1, as the step applies it."""
    out = np.zeros((n, T, 3), np.float32)
    rc = lib().push_sample(C.byref(params), int(seed) & (2 ** 64 - 1), int(gid0), int(n), int(episode), int(t0),
                           int(T), out.ctypes.data_as(C.POINTER(C.c_float)))
    if rc != 0:
        raise ValueError(f"push_sample rejected the push fields (rc {rc})")
    return out
