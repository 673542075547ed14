"""TEST INFRASTRUCTURE — ctypes binding of oracle/risk6_vector.c: the six-player search with a six-seat value vector (SIXPLAYER.md §2),
the checker of az_mcts6_* over a network with six value outputs or with the AZ_EVAL_PSEUDO6 evaluator.

The library is compiled on first use, with the flags of oracle/Makefile, into a private temporary directory (the tree may be read-only).
Games are pyoracle.Oracle6Game objects and rules pyoracle.RoRules, as for lockstep6.Lockstep6Mcts."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "risk_oracle.c"), os.path.join(HERE, "risk6_vector.c")]
# evaluator callback: (state, policy[43] out, value[6] out, user)
EVAL6_CB = C.CFUNCTYPE(None, C.POINTER(po.R6State), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p)
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="risk6_vector_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "librisk6_vector.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-std=gnu99", "-O2", "-fPIC", "-Wall", "-Wextra", "-ffp-contract=off",
                               "-I" + HERE, "-I" + os.path.join(os.path.dirname(HERE), "include"), "-shared", "-o", so] + SOURCES + ["-lm"])
        L = C.CDLL(so)
        f32 = np.ctypeslib.ndpointer(np.float32, flags="C")
        L.r6v_new.restype = C.c_void_p
        L.r6v_new.argtypes = [C.c_void_p, C.c_void_p]
        L.r6v_free.argtypes = [C.c_void_p]
        L.r6v_table_size.argtypes = [C.c_void_p]
        for fn in ("r6v_vl_skips", "r6v_active_total"):
            getattr(L, fn).argtypes = [C.c_void_p]
            getattr(L, fn).restype = C.c_uint64
        L.r6v_eval_pseudo6.argtypes = [C.POINTER(po.R6State), f32, f32, C.c_void_p]
        L.r6v_search.argtypes = [C.c_void_p, C.POINTER(po.R6State), C.POINTER(po.RoRules), C.c_uint64, C.c_uint32, C.c_uint32, C.c_int,
                                 np.ctypeslib.ndpointer(np.uint32, flags="C"), f32, f32, f32, C.POINTER(C.c_uint32), C.POINTER(C.c_float)]
        _lib = L
    return _lib


def pseudo6(game_obj):
    """(policy[43], value[6]) of the C pseudo6 evaluator at a position"""
    p, v = np.zeros(po.MOVES, np.float32), np.zeros(6, np.float32)
    lib().r6v_eval_pseudo6(C.byref(game_obj.s), p, v, None)
    return p, v


class Vector6Mcts:
    """one tree of the value-vector search (table cleared per search; the pseudo6 evaluator unless `eval_fn`, an EVAL6_CB, is given)"""

    def __init__(self, rules=None, eval_fn=None):
        self.L = lib()
        self.rules = rules if rules is not None else po.default_rules()
        self._keep = eval_fn
        self.h = self.L.r6v_new(C.cast(eval_fn, C.c_void_p) if eval_fn is not None else None, None)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.r6v_free(self.h)
            self.h = None

    def table_size(self):
        return int(self.L.r6v_table_size(self.h))

    def vl_skips(self):
        return int(self.L.r6v_vl_skips(self.h))

    def active_total(self):
        """the sum of the table's active_N marks (0 after a completed search)"""
        return int(self.L.r6v_active_total(self.h))

    def search_rc(self, game_obj, seed, game, ply, lockstep):
        N = np.zeros(po.MOVES, np.uint32)
        Q, P, pi = (np.zeros(po.MOVES, np.float32) for _ in range(3))
        sumN, val = C.c_uint32(0), C.c_float(0)
        rc = self.L.r6v_search(self.h, C.byref(game_obj.s), C.byref(self.rules), seed, game, ply, int(lockstep), N, Q, P, pi,
                               C.byref(sumN), C.byref(val))
        return rc, dict(N=N, Q=Q, P=P, pi=pi, sumN=int(sumN.value), value=float(val.value))

    def search(self, game_obj, seed, game, ply, lockstep=1):
        rc, out = self.search_rc(game_obj, seed, game, ply, lockstep)
        assert rc == 0, rc
        return out

    def pick(self, pi, sample, seed, game, ply):
        return int(po.oracle_lib().ro_pick_move(np.ascontiguousarray(pi, np.float32), int(sample), seed, game, ply))
