"""CPU suite of the six-player scripted agent (SIXPLAYER.md §5) on its oracle (oracle/risk6_script.c through oracle/script6.py):
legal in every position of games through eliminations under every rule set, a pure function of the position, each clause pinned by a
hand-built position, games between scripts finish, and the script beats the uniform-random player."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import pyoracle as po
from oracle import script6 as s6

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0x5EED0006
RUNNING, DRAW = -1, -2
RULE_SETS = [dict(), dict(limit_attack=1), dict(limit_reinforcement=0), dict(allow_yield=0, max_game_rounds=30), dict(min_unit_move=1)]
RULE_IDS = ["default", "limit_attack", "no_limit_reinf", "no_yield_30_rounds", "min_unit_move_1"]


def play(rules, deal, game, script_agent, rot=0, check=None):
    """one game from the deal of game id `deal` with all randomness keyed by `game`: seat s is agent (s + rot) % 6, the agents in
    script_agent play the script, the others the random player; check(o, action) sees every scripted position before its move.
    Returns (status, plies, the fewest seats alive at any point)"""
    o = po.Oracle6Game(rules)
    o.new_game(SEED, deal, 0)
    ply, alive = 0, 6
    while o.status() == RUNNING:
        if (o.s.cur + rot) % 6 in script_agent:
            a = s6.script_action(o)
            if check:
                check(o, a)
        else:
            a = o.random_action(SEED, game, ply)
        assert o.move(a, SEED, game, ply) == 0
        ply += 1
        alive = min(alive, len(set(o.s.owner)))
    return o.status(), ply, alive


@pytest.mark.parametrize("kw", RULE_SETS, ids=RULE_IDS)
def test_legal_in_every_phase_through_eliminations(kw):
    rules = po.default_rules(**kw)
    seen = set()

    def check(o, a):
        assert 0 <= a <= po.SKIP and (o.valid() >> a) & 1, (a, bytes(o.s).hex())
        seen.add((int(o.s.phase), a == po.SKIP))

    fewest = 6
    for g in range(8):
        fewest = min(fewest, play(rules, 100 + g, 100 + g, {0, 2, 4}, rot=g % 6, check=check)[2])
    assert fewest < 6                                            # seats were eliminated
    assert {p for p, _ in seen} == {0, 2, 3, 4, 5}
    assert (3, False) in seen and (5, False) in seen
    if not kw.get("limit_attack"):
        assert (3, True) in seen


def test_pure_function_of_the_position():
    o = po.Oracle6Game()
    o.new_game(SEED, 7, 0)
    ply = 0
    while o.status() == RUNNING:
        before = bytes(o.s)
        a = s6.script_action(o)
        assert bytes(o.s) == before
        copy = po.Oracle6Game()
        copy.set_image(np.frombuffer(before, np.uint8))
        assert s6.script_action(copy) == a == s6.script_action(o)
        assert o.move(a if ply % 3 else o.random_action(SEED, 7, ply), SEED, 7, ply) == 0
        ply += 1


@pytest.mark.parametrize("case", s6.HAND_CASES, ids=[c[0] for c in s6.HAND_CASES])
def test_hand_built_positions(case):
    name, kw, rules_kw, want = case
    o = s6.position(**kw)
    o.rules = po.default_rules(**rules_kw)
    assert o.status() == RUNNING
    a = s6.script_action(o)
    assert a == want, (name, a)
    assert (o.valid() >> a) & 1


@pytest.mark.parametrize("kw", [dict(), dict(allow_yield=0, max_game_rounds=30)], ids=["default", "no_yield_30_rounds"])
def test_script_only_games_finish(kw):
    rules = po.default_rules(**kw)
    for g in range(6):
        st, plies, _ = play(rules, 300 + g, 300 + g, set(range(6)))
        assert st != RUNNING and plies > 78


def test_script_beats_random_players():
    """120 seat-rotated games (20 deals, the script in each seat of each deal once), 1 script vs 5 random players, default rules"""
    rules = po.default_rules()
    wins = 0
    for g in range(120):
        r = g % 6
        st, _, _ = play(rules, g - r, g, {0}, rot=r)
        wins += st != DRAW and (st + r) % 6 == 0
    assert wins >= 100, wins


def test_constants_agree_with_the_headers():
    L = s6.lib()
    assert (L.r6s_margin(), L.r6s_fortify_below()) == (s6.MARGIN, s6.FORTIFY_BELOW)
    cuh = open(os.path.join(ROOT, "alphazero_risk_b200", "csrc", "az_script6.cuh")).read()
    assert int(re.search(r"#define E6_SCRIPT_MARGIN (\d+)", cuh).group(1)) == s6.MARGIN
    assert int(re.search(r"#define E6_SCRIPT_FORTIFY_BELOW (\d+)", cuh).group(1)) == s6.FORTIFY_BELOW
    masks = re.search(r"E6_CONT_MASK\[6\] = \{(.*?)\}", cuh).group(1)
    want = (C.c_uint64 * 6).in_dll(po.oracle_lib(), "RO_CONTINENT_MASK")
    assert [int(v.strip().rstrip("ull"), 16) for v in masks.split(",")] == list(want)
    h = open(os.path.join(ROOT, "include", "az_b200.h")).read()
    from alphazero_risk_b200 import api
    for name in ("SEARCHER", "RANDOM", "SCRIPT"):
        assert int(re.search(r"#define AZ_AGENT6_%s (\d+)" % name, h).group(1)) == getattr(api, "AGENT6_" + name)
