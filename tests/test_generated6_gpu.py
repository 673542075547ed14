"""GPU suite of the generated six-player games (az_env6_play / az_env6_record / az_env6_samples, SIXPLAYER.md §6).  The checker is
oracle/generated6.py on the C oracle: state images and counters bit for bit, and the record queue byte for byte as whole per-game
blocks in any order."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as po
from oracle.generated6 import Generated6

pytestmark = pytest.mark.gpu
SEED = 0x5EED0006
REC = 288
ALL = 0x3f


@pytest.fixture(scope="module")
def api():
    from alphazero_risk_b200 import api as a
    if a.lib().az_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu suite must run on a B200")
    return a


def kinds(api, script):
    return [api.SCRIPT6 if (script >> s) & 1 else None for s in range(6)]


def match_whole_games(recs, expected):
    """the queue = whole expected games back to back (in any order); returns the games found"""
    blob, left, pos, found = recs.tobytes(), sorted(expected, key=len, reverse=True), 0, []
    while pos < len(blob):
        hit = [e for e in left if blob.startswith(e, pos)]
        assert hit, "record stream at byte %d matches no expected game" % pos
        left.remove(hit[0]); found.append(hit[0]); pos += len(hit[0])
    return found


def row_multiset(recs):
    return np.sort(np.ascontiguousarray(recs).view(np.dtype((np.void, REC))).reshape(-1))


@pytest.mark.parametrize("kw", [dict(), dict(allow_yield=0, max_game_rounds=30)], ids=["default", "no_yield_30_rounds"])
def test_random_play_is_the_rollout(api, kw):
    n, steps, first, a = 128, 3500, 40, 1300
    rules = api.default_rules(**kw)
    out = []
    for how in ("rollout", "play_split", "play_once", "play_recording_env"):
        env = api.Env6(n, rules=rules, first_game_id=first)
        env.reset(SEED)
        if how == "rollout":
            env.rollout(a); env.rollout(steps - a)
        elif how == "play_split":
            env.play([None] * 6, a); env.play([None] * 6, steps - a)
        elif how == "play_once":
            env.play([None] * 6, steps)
        else:                                   # recording enabled: k_env6_play's own random player, nothing recorded
            env.record(capacity_samples=1000, max_samples_per_game=64)
            env.play([None] * 6, a); env.play([None] * 6, steps - a)
            assert len(env.samples()[0]) == 0
        out.append((env.export(), env.counters()))
        env.close()
    (i0, c0) = out[0]
    for i, c in out[1:]:
        assert (i0 == i).all() and c0 == c
    assert c0["steps"] == n * steps and c0["games"] > n // 2


CONFIGS = [(ALL, ALL, {}), (0x01, 0x01, {}), (0x15, ALL, {}), (0x09, ALL, dict(limit_attack=1))]
CONFIG_IDS = ["six_scripts", "one_script_recorded", "scripts_0_2_4", "limit_attack"]
N2, FIRST2, PLIES2, SPLIT2 = 128, 900, 2400, 1500


@pytest.mark.parametrize("script,record_seats,kw", CONFIGS, ids=CONFIG_IDS)
def test_mixed_kinds_match_oracle(api, script, record_seats, kw):
    """two calls (games running across the boundary keep their staged samples) against the oracle replay"""
    env = api.Env6(N2, rules=api.default_rules(**kw), first_game_id=FIRST2)
    env.reset(SEED)
    env.record(capacity_samples=N2 * PLIES2, max_samples_per_game=4096)
    env.play(kinds(api, script), SPLIT2, record_seats)
    r1, d1 = env.samples()
    env.play(kinds(api, script), PLIES2 - SPLIT2, record_seats)
    r2, d2 = env.samples()
    img, cnt = env.export(), env.counters()
    env.close()
    o = Generated6(N2, FIRST2, SEED, po.default_rules(**kw))
    e1 = o.play(script, record_seats, SPLIT2)
    e2 = o.play(script, record_seats, PLIES2 - SPLIT2)
    assert (img == o.images()).all()
    assert cnt == o.counters and cnt["games"] >= N2
    assert d1 == 0 and d2 == 0 and len(e1) >= N2 // 2 and len(e2) > 0
    for recs, exp in ((r1, e1), (r2, e2)):
        assert sum(len(e) for e in exp) == recs.size
        assert len(match_whole_games(recs, exp)) == len(exp)
    assert set(np.unique(np.concatenate([r1, r2])[:, 98])) <= {s for s in range(6) if (record_seats >> s) & 1}


def test_unrecorded_call_queues_the_games_it_ends(api):
    """a call with record_seats = 0 on a recording env still queues the blocks of games that end in it (their samples come from an
    earlier call) and leaves nothing of them staged for the next game"""
    n, first, script = 64, 400, 0x15
    calls = [(ALL, 400), (0, 900), (ALL, 1200), (0x06, 700)]
    env = api.Env6(n, first_game_id=first)
    env.reset(SEED)
    env.record(capacity_samples=n * 3200, max_samples_per_game=4096)
    o = Generated6(n, first, SEED)
    for seats, plies in calls:
        env.play(kinds(api, script), plies, seats)
        recs, dropped = env.samples()
        exp = o.play(script, seats, plies)
        assert dropped == 0 and len(exp) > 0, (seats, plies)
        assert sum(len(e) for e in exp) == recs.size
        assert len(match_whole_games(recs, exp)) == len(exp)
    assert (env.export() == o.images()).all() and env.counters() == o.counters
    env.close()


def test_recording_changes_nothing(api):
    n, plies, script = 96, 1700, 0x15
    out = []
    for mode in ("off", "enabled_no_seats", "all_seats"):
        env = api.Env6(n, first_game_id=11)
        env.reset(SEED)
        if mode != "off":
            env.record(capacity_samples=n * plies, max_samples_per_game=2048)
        for part in (600, plies - 600):
            env.play(kinds(api, script), part, ALL if mode == "all_seats" else 0)
        recs = env.samples()[0] if mode != "off" else None
        out.append((env.export(), env.counters(), recs))
        env.close()
    (i0, c0, _), (i1, c1, r1), (i2, c2, r2) = out
    assert (i0 == i1).all() and (i0 == i2).all() and c0 == c1 == c2 and c0["games"] > 0
    assert len(r1) == 0 and len(r2) > 0


N4, FIRST4, PLIES4, SCRIPT4 = 48, 3, 1800, 0x2d


@pytest.fixture(scope="module")
def expected4():
    return Generated6(N4, FIRST4, SEED).play(SCRIPT4, ALL, PLIES4)


def played(api, capacity, max_per_game):
    env = api.Env6(N4, first_game_id=FIRST4)
    env.reset(SEED)
    env.record(capacity_samples=capacity, max_samples_per_game=max_per_game)
    env.play(kinds(api, SCRIPT4), PLIES4, ALL)
    recs, dropped = env.samples()
    again = env.samples()
    env.close()
    return recs, dropped, again


def test_small_queue_returns_whole_games_and_counts_the_rest(api, expected4):
    total = sum(len(e) for e in expected4) // REC
    cap = total // 3
    recs, dropped, again = played(api, cap, 4096)
    assert 0 < len(recs) <= cap
    found = match_whole_games(recs, expected4)
    assert sum(len(f) for f in found) == recs.size
    assert len(recs) + dropped == total
    assert len(again[0]) == 0 and again[1] == 0            # the drain reset the dropped count


def test_game_longer_than_staging_is_dropped_whole(api, expected4):
    lengths = sorted(len(e) // REC for e in expected4)
    limit = lengths[len(lengths) // 2]
    recs, dropped, _ = played(api, N4 * PLIES4, limit)
    kept = [e for e in expected4 if len(e) // REC <= limit]
    assert 0 < len(kept) < len(expected4)
    assert sorted(match_whole_games(recs, expected4)) == sorted(kept)
    assert dropped == sum(len(e) // REC for e in expected4 if len(e) // REC > limit)


def test_size_query_and_drain(api, expected4):
    """az_env6_samples: h_records = NULL is a size query that leaves the queue alone; a drain empties it and resets the dropped count"""
    total = sum(len(e) for e in expected4) // REC
    env = api.Env6(N4, first_game_id=FIRST4)
    env.reset(SEED)
    env.record(capacity_samples=total - 1, max_samples_per_game=4096)
    env.play(kinds(api, SCRIPT4), PLIES4, ALL)
    L, n, dropped = env.L, C.c_size_t(0), C.c_uint64(0)
    for _ in range(2):
        api.check(L.az_env6_samples(env.h, None, C.c_size_t(0), C.byref(n), C.byref(dropped), None))
        assert 0 < n.value < total and dropped.value > 0 and n.value + dropped.value == total
    have = n.value
    small = np.empty((have - 1, REC), np.uint8)
    assert L.az_env6_samples(env.h, api._ptr(small), C.c_size_t(have - 1), C.byref(n), C.byref(dropped), None) != 0
    out = np.empty((have, REC), np.uint8)
    api.check(L.az_env6_samples(env.h, api._ptr(out), C.c_size_t(have), C.byref(n), C.byref(dropped), None))
    assert n.value == have
    assert len(match_whole_games(out, expected4)) > 0
    api.check(L.az_env6_samples(env.h, None, C.c_size_t(0), C.byref(n), C.byref(dropped), None))
    assert n.value == 0 and dropped.value == 0
    env.close()


def test_running_game_keeps_its_samples_across_calls(api):
    """plies played one call at a time: no game has ended after the set-up, so nothing is queued; the first finished games then
    come out whole, with the samples of every call"""
    n, first = 16, 70
    env = api.Env6(n, first_game_id=first)
    env.reset(SEED)
    env.record(capacity_samples=200000, max_samples_per_game=4096)
    o = Generated6(n, first, SEED)
    got, exp = [], []
    for step in (1, 5, 72, 200, 7, 900, 1):
        env.play(kinds(api, ALL), step, ALL)
        exp += o.play(ALL, ALL, step)
        r, dropped = env.samples()
        assert dropped == 0
        if step in (1, 5, 72):
            assert len(r) == 0
        got.append(r)
    recs = np.concatenate(got)
    assert len(exp) > 0 and sum(len(e) for e in exp) == recs.size
    assert len(match_whole_games(recs, exp)) == len(exp)
    assert (env.export() == o.images()).all()
    env.close()


@pytest.mark.parametrize("how", ["reset", "import"])
def test_reset_or_import_discards_staged_samples(api, how):
    n, first, pre, plies = 32, 60, 200, 1500
    env = api.Env6(n, first_game_id=first)
    env.reset(SEED)
    env.record(capacity_samples=n * plies, max_samples_per_game=4096)
    env.play(kinds(api, ALL), pre, ALL)                       # set-up and the first rounds: no game has ended
    assert len(env.samples()[0]) == 0
    seed = SEED + 7 if how == "reset" else SEED
    o = Generated6(n, first, seed)
    if how == "reset":
        env.reset(seed)
    else:
        env.import_images(env.export())
        o.play(ALL, 0, pre)                                  # the same plies, nothing staged
    env.play(kinds(api, ALL), plies, ALL)
    recs, dropped = env.samples()
    expected = o.play(ALL, ALL, plies)
    assert dropped == 0 and len(expected) >= n // 2
    assert sum(len(e) for e in expected) == recs.size
    assert len(match_whole_games(recs, expected)) == len(expected)
    env.close()


def test_full_size_properties(api):
    """configs[3]'s game count: reproducible, shard invariant, a sampled oracle replay"""
    n, plies, script, seats = 16384, 700, 0x15, 0x03
    rules = api.default_rules(max_game_rounds=20)

    def run(count, first):
        env = api.Env6(count, rules=rules, first_game_id=first)
        env.reset(SEED)
        env.record(capacity_samples=count * 300, max_samples_per_game=1024)
        env.play(kinds(api, script), 300, seats)
        env.play(kinds(api, script), plies - 300, seats)
        recs, dropped = env.samples()
        out = (env.export(), env.counters(), recs, dropped)
        env.close()
        return out

    img, cnt, recs, dropped = run(n, 0)
    img2, cnt2, recs2, _ = run(n, 0)
    assert dropped == 0 and cnt["steps"] == n * plies and cnt["games"] > n // 2
    assert (img == img2).all() and cnt == cnt2 and (row_multiset(recs) == row_multiset(recs2)).all()
    lo, hi = run(n // 2, 0), run(n // 2, n // 2)
    assert (np.concatenate([lo[0], hi[0]]) == img).all()
    assert (row_multiset(np.concatenate([lo[2], hi[2]])) == row_multiset(recs)).all()
    ids = sorted(int(g) for g in np.random.default_rng(3).choice(n, 32, replace=False))
    o = Generated6(0, 0, SEED, po.default_rules(max_game_rounds=20), game_ids=ids)
    exp = o.play(script, seats, 300) + o.play(script, seats, plies - 300)
    assert (img[ids] == o.images()).all()
    blob = recs.tobytes()
    assert len(exp) >= 16
    for e in exp:
        at = blob.find(e)
        assert at >= 0 and at % REC == 0


@pytest.mark.parametrize("planes,vo", [(13, 1), (16, 1), (13, 6), (16, 6)])
def test_train6_on_generated_records(api, planes, vo):
    env = api.Env6(256, rules=api.default_rules(max_game_rounds=20), first_game_id=5)
    env.reset(SEED)
    env.record(capacity_samples=256 * 1500, max_samples_per_game=2048)
    env.play(kinds(api, ALL), 1500, ALL)
    recs, dropped = env.samples()
    env.close()
    assert dropped == 0 and len(recs) >= 20000
    net = api.Net(blocks=1, seed=7, value_outputs=vo, input_planes=planes)
    lp, lv = net.train6(recs[:20480], epochs=3, batch_size=256, seed=11)
    net.close()
    assert np.isfinite(lp).all() and np.isfinite(lv).all()
    assert lp[2] < lp[1] < lp[0], lp


def test_rejections(api):
    env = api.Env6(8)
    env.reset(SEED)
    L = env.L
    good = api._ptr(np.full(6, api.AGENT6_RANDOM, np.int32))
    n, dropped = C.c_size_t(0), C.c_uint64(0)
    assert L.az_env6_samples(env.h, None, C.c_size_t(0), C.byref(n), C.byref(dropped), None) != 0          # before az_env6_record
    assert L.az_env6_play(env.h, good, 1, 10, None) != 0                                                  # record_seats without record
    for bad in (api.AGENT6_SEARCHER, 3, -1):
        k = np.array([api.AGENT6_SCRIPT] * 5 + [bad], np.int32)
        assert L.az_env6_play(env.h, api._ptr(k), 0, 10, None) != 0
    assert L.az_env6_play(env.h, None, 0, 10, None) != 0
    assert L.az_env6_play(env.h, good, 0, -1, None) != 0
    assert L.az_env6_record(env.h, C.c_size_t(0), 16) != 0
    assert L.az_env6_record(env.h, C.c_size_t(100), 0) != 0
    assert L.az_env6_record(env.h, C.c_size_t(100), -3) != 0
    env.record(1000, 64)
    assert L.az_env6_record(env.h, C.c_size_t(100), 16) != 0                                               # already enabled
    for seats in (64, 65, 0xffffffff):
        assert L.az_env6_play(env.h, good, seats, 10, None) != 0
    with pytest.raises(api.AzError):
        env.play([None] * 5 + [object()], 10)
    for seats in (64, -1, 1 << 32, (1 << 32) + 1):
        with pytest.raises(api.AzError):
            env.play([None] * 6, 10, seats)
    img = env.export()
    assert env.counters()["steps"] == 0 and (img == env.export()).all()
    env.play([None] * 6, 0, ALL)
    env.play([api.SCRIPT6] * 6, 10, 63)
    assert env.counters()["steps"] == 80
    env.close()
