"""TEST INFRASTRUCTURE — ctypes binding of oracle/risk6_planes.c: the six-player seat planes (SIXPLAYER.md §2), the 16-plane network
input: the checker of az_env6_encode_planes(16) and of the six-player search over a 16-plane network.

The library is compiled on first use, with the flags of oracle/Makefile, into a private temporary directory (the tree may be read-only).
Games are pyoracle.Oracle6Game objects."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "risk_oracle.c"), os.path.join(HERE, "risk6_planes.c")]
INPUT6_FLOATS = 672          # [7][6][16], R6_INPUT16_FLOATS
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="risk6_planes_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "librisk6_planes.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-std=gnu99", "-O2", "-fPIC", "-Wall", "-Wextra", "-ffp-contract=off",
                               "-I" + HERE, "-I" + os.path.join(os.path.dirname(HERE), "include"), "-shared", "-o", so] + SOURCES + ["-lm"])
        L = C.CDLL(so)
        L.r6_encode16.argtypes = [C.POINTER(po.R6State), np.ctypeslib.ndpointer(np.float32, flags="C")]
        L.r6_encode.argtypes = [C.POINTER(po.R6State), np.ctypeslib.ndpointer(np.float32, flags="C")]
        assert C.c_int.in_dll(L, "r6_input16_floats").value == INPUT6_FLOATS
        _lib = L
    return _lib


def encode16_state(state_ptr):
    """the 16 seat planes of an R6State pointer (an evaluator callback's argument), [672]"""
    x = np.zeros(INPUT6_FLOATS, np.float32)
    lib().r6_encode16(state_ptr, x)
    return x


def encode16(game_obj):
    """the 16 seat planes of a pyoracle.Oracle6Game position, [672] = [7][6][16]"""
    return encode16_state(C.byref(game_obj.s))


def encode13(game_obj):
    """r6_encode (the 13-plane six-seat input) of the same library, [546]"""
    x = np.zeros(po.INPUT_FLOATS, np.float32)
    lib().r6_encode(C.byref(game_obj.s), x)
    return x
