"""TEST INFRASTRUCTURE — ctypes binding of oracle/risk6_script.c: the six-player scripted agent of SIXPLAYER.md §5, the checker of
az_env6_script_actions and of the scripted agents of az_arena6_*.

The library is compiled on first use, with the flags of oracle/Makefile, into a private temporary directory (the tree may be read-only).
Games are pyoracle.Oracle6Game objects and rules pyoracle.RoRules."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "risk_oracle.c"), os.path.join(HERE, "risk6_script.c")]
MARGIN = 2              # R6S_MARGIN: an optional attack needs a source at least this many armies above its target
FORTIFY_BELOW = 32      # R6S_FORTIFY_BELOW: a fortify target holds fewer armies than this
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="risk6_script_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "librisk6_script.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-std=gnu99", "-O2", "-fPIC", "-Wall", "-Wextra", "-ffp-contract=off",
                               "-I" + HERE, "-I" + os.path.join(os.path.dirname(HERE), "include"), "-shared", "-o", so] + SOURCES + ["-lm"])
        L = C.CDLL(so)
        L.r6_script_action.argtypes = [C.POINTER(po.R6State), C.POINTER(po.RoRules)]
        _lib = L
    return _lib


def script_action(game_obj, rules=None):
    """the scripted action of the position of `game_obj` (a pyoracle.Oracle6Game) under `rules` (default: the game's own)"""
    return int(lib().r6_script_action(C.byref(game_obj.s), C.byref(rules if rules is not None else game_obj.rules)))


def position(own, army=None, phase=3, cur=0, mob=(po.NONE, po.NONE), reinf=0):
    """a running six-player position: seat `cur` owns the lands of `own`, every other land i belongs to seat (cur + 1 + i % 5) % 6;
    every land holds one army unless `army` ({land: armies}) says otherwise; no cards, no set-up pool, round 3"""
    o = po.Oracle6Game()
    s = o.s
    for i in range(po.LANDS):
        s.owner[i] = cur if i in own else (cur + 1 + i % 5) % 6
        s.army[i] = (army or {}).get(i, 1)
    s.round, s.cur, s.phase, s.reinf = 3, cur, phase, reinf
    s.mob_from, s.mob_to = mob
    return o


# hand-built positions that pin the clauses of SIXPLAYER.md §5: (name, position kwargs, rules kwargs, the scripted action).
# Continents: NA 0..8, SA 9..12, EU 13..19, AF 20..25, AS 26..37, AU 38..41.
HAND_CASES = [
    # attack: SA (one foreign land) before NA although 8 and 11 have the same margin and 8 is the lower index
    ("attack_fewest_foreign_continent", dict(own={9, 10, 12}, army={9: 5, 10: 5}), {}, 11),
    # attack: SA and AU both have two foreign lands; AU has more attackable ones (SA's 12 is out of reach), its weakest is 41
    ("attack_tie_more_targets", dict(own={9, 10, 38, 39}, army={9: 6, 38: 6, 39: 6, 40: 3, 41: 2}), {}, 41),
    # attack: SA and AU tie on both counts: the lower continent index, then the larger margin / lower land (11 over 12)
    ("attack_tie_lowest_continent", dict(own={9, 10, 38, 39}, army={9: 6, 10: 6, 38: 6, 39: 6, 40: 3, 41: 2}), {}, 11),
    # attack: margin 2 attacks, margin 1 skips, margin 1 under limit_attack (SKIP illegal) attacks
    ("attack_margin_2", dict(own={41}, army={41: 4, 39: 2, 40: 2}), {}, 39),
    ("attack_margin_1_skips", dict(own={41}, army={41: 3, 39: 2, 40: 2}), {}, 42),
    ("attack_forced_by_limit_attack", dict(own={41}, army={41: 3, 39: 2, 40: 2}), dict(limit_attack=1), 39),
    # attack: the target continent's best margin is 1, so the largest margin anywhere (4, lowest land 9) is played instead
    ("attack_margin_elsewhere", dict(own={40, 41, 11}, army={41: 2, 11: 5}), {}, 9),
    # reinforcement: target 40 (AU); its neighbours 38 and 39 tie at 3 armies, 39 comes first in 40's neighbour list
    ("reinforce_strongest_neighbour_order", dict(own={38, 39}, army={38: 3, 39: 3, 41: 2}, phase=2, reinf=6), {}, 39),
    # reinforcement: AU's targets touch only full lands, so the land facing the most foreign armies (12: 5 + 5) is played
    ("reinforce_no_strongest", dict(own={0, 12, 38, 39}, army={38: 32, 39: 32, 10: 5, 11: 5}, phase=2, reinf=6), {}, 12),
    # set-up: the same rule as reinforcement
    ("setup_strongest_neighbour_order", dict(own={38, 39}, army={38: 3, 39: 3, 41: 2}, phase=0), {}, 39),
    # mobilisation: stop (play mob_from) when the destination is interior and the source borders a foreign land, else continue
    ("mobilize_stop", dict(own={39, 40, 41}, army={40: 5, 41: 2}, phase=4, mob=(40, 41)), {}, 40),
    ("mobilize_continue", dict(own={39, 40, 41}, army={40: 5, 39: 2}, phase=4, mob=(40, 39)), {}, 39),
    # fortify: border lands 39 and 40 face 38's 7 armies; 40 holds fewer, so it scores higher
    ("fortify_target", dict(own={39, 40, 41}, army={38: 7, 39: 3, 40: 2, 41: 9}, phase=5), {}, 40),
    ("fortify_skips_full", dict(own={39, 40, 41}, army={38: 7, 39: 3, 40: 32, 41: 9}, phase=5), {}, 39),
    ("fortify_skip", dict(own={39, 40, 41}, army={38: 7, 39: 32, 40: 32, 41: 9}, phase=5), {}, 42),
]
