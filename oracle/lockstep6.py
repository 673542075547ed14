"""TEST INFRASTRUCTURE — ctypes binding of oracle/risk6_lockstep.c: the six-player search with K descents per round under the active_N
rule (SIXPLAYER.md §2), the checker of az_mcts6_* with az_rules.concurrent_descents = K.

The library is compiled on first use, with the flags of oracle/Makefile, into a private temporary directory (the tree may be read-only).
Games are pyoracle.Oracle6Game objects and rules pyoracle.RoRules, as for pyoracle.Oracle6Mcts."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "risk_oracle.c"), os.path.join(HERE, "risk6_lockstep.c")]
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="risk6_lockstep_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "librisk6_lockstep.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-std=gnu99", "-O2", "-fPIC", "-Wall", "-Wextra", "-ffp-contract=off",
                               "-I" + HERE, "-I" + os.path.join(os.path.dirname(HERE), "include"), "-shared", "-o", so] + SOURCES + ["-lm"])
        L = C.CDLL(so)
        f32 = np.ctypeslib.ndpointer(np.float32, flags="C")
        L.r6l_new.restype = C.c_void_p
        L.r6l_new.argtypes = [C.c_void_p, C.c_void_p]
        L.r6l_free.argtypes = [C.c_void_p]
        L.r6l_table_size.argtypes = [C.c_void_p]
        for fn in ("r6l_vl_skips", "r6l_vl_duplicates", "r6l_active_total"):
            getattr(L, fn).argtypes = [C.c_void_p]
            getattr(L, fn).restype = C.c_uint64
        L.r6l_search.argtypes = [C.c_void_p, C.POINTER(po.R6State), C.POINTER(po.RoRules), C.c_uint64, C.c_uint32, C.c_uint32, C.c_int,
                                 np.ctypeslib.ndpointer(np.uint32, flags="C"), f32, f32, f32, C.POINTER(C.c_uint32), C.POINTER(C.c_float)]
        _lib = L
    return _lib


class Lockstep6Mcts:
    """one tree of the lockstep search (table cleared per search; pseudo evaluator unless `eval_fn` is given)"""

    def __init__(self, rules=None, eval_fn=None):
        self.L = lib()
        self.rules = rules if rules is not None else po.default_rules()
        self._keep = eval_fn
        self.h = self.L.r6l_new(C.cast(eval_fn, C.c_void_p) if eval_fn is not None else None, None)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.r6l_free(self.h)
            self.h = None

    def table_size(self):
        return int(self.L.r6l_table_size(self.h))

    def vl_counts(self):
        """(moves passed over by the active_N rule, duplicate requests) so far"""
        return int(self.L.r6l_vl_skips(self.h)), int(self.L.r6l_vl_duplicates(self.h))

    def active_total(self):
        """the sum of the table's active_N marks (0 after a completed search)"""
        return int(self.L.r6l_active_total(self.h))

    def search_rc(self, game_obj, seed, game, ply, lockstep):
        N = np.zeros(po.MOVES, np.uint32)
        Q, P, pi = (np.zeros(po.MOVES, np.float32) for _ in range(3))
        sumN, val = C.c_uint32(0), C.c_float(0)
        rc = self.L.r6l_search(self.h, C.byref(game_obj.s), C.byref(self.rules), seed, game, ply, int(lockstep), N, Q, P, pi,
                               C.byref(sumN), C.byref(val))
        return rc, dict(N=N, Q=Q, P=P, pi=pi, sumN=int(sumN.value), value=float(val.value))

    def search(self, game_obj, seed, game, ply, lockstep=1):
        rc, out = self.search_rc(game_obj, seed, game, ply, lockstep)
        assert rc == 0, rc
        return out

    def pick(self, pi, sample, seed, game, ply):
        return int(po.oracle_lib().ro_pick_move(np.ascontiguousarray(pi, np.float32), int(sample), seed, game, ply))
