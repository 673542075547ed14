"""Self-play training samples (SURVEY.md 8f N3): record layout and file format against the reference's own
NNInputData / NNTrainDataStorage, then the device-side recording against an oracle replay of the same games."""
import os

import numpy as np
import pytest

from oracle import pyoracle as po

SEED = 0x5EED0001
NEED_REF = pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref not built (needs /root/reference)")


def random_positions(game_cls, n_games, steps):
    """(game object after k random-play steps) snapshots, reproducible"""
    out = []
    for g in range(n_games):
        o = game_cls()
        o.new_game(SEED, g, 0)
        for ply in range(steps):
            if o.status() != -1:
                break
            if ply % 7 == 3:
                out.append((g, ply, o.data().copy()))
            assert o.move(o.random_action(SEED, g, ply), SEED, g, ply) == 0
    return out


@NEED_REF
def test_nn_input_image_matches_reference():
    """ro_nn_input == the bytes of the reference's NNInputData(const State&) (padding bytes 43, 46, 47 excluded)"""
    snaps = random_positions(po.RefGame, 6, 400)
    assert len(snaps) > 200
    ref, orc = po.RefGame(), po.OracleGame()
    keep = np.ones(88, bool); keep[[43, 46, 47]] = False
    for _, _, data in snaps:
        ref.set_data(data); assert orc.set_data(data) == 0
        assert (ref.nn_input()[keep] == orc.nn_input()[keep]).all()
        assert (orc.nn_input()[~keep] == 0).all()


@NEED_REF
def test_samples_file_is_the_reference_format(tmp_path):
    """az_samples_write_file writes byte for byte what NNTrainDataStorage::saveTrainingSamples writes"""
    from alphazero_risk_b200 import api
    rng = np.random.default_rng(5)
    snaps = random_positions(po.OracleGame, 3, 300)[:64]
    orc = po.OracleGame()
    for status in (0, 1, -2):
        players, inputs, pols, recs = [], [], [], []
        for _, _, data in snaps:
            assert orc.set_data(data) == 0
            pi = rng.random(43, dtype=np.float32); pi /= pi.sum()
            players.append(orc.s.cur); inputs.append(orc.nn_input()); pols.append(pi)
            recs.append(orc.sample_record(pi, status))
        ref_path, our_path = str(tmp_path / ("ref%d.bin" % status)), str(tmp_path / ("ours%d.bin" % status))
        po.ref_save_samples(ref_path, players, np.stack(inputs), np.stack(pols), status, 40)
        api.write_samples_file(our_path, np.stack(recs))
        a, b = open(ref_path, "rb").read(), open(our_path, "rb").read()
        assert len(a) == 8 + 265 * len(snaps) and a == b


def test_samples_file_matches_the_reference_bytes(golden_dir, tmp_path):
    """az_samples_write_file around the records the reference's NNTrainDataStorage::saveTrainingSamples wrote (tests/golden/
    turn_samples.npz, generator tests/golden/gen_turn_samples.py): the reference's file is the record count as uint64, then the
    265-byte records, so writing those records must give back exactly that file"""
    from alphazero_risk_b200 import api
    z = np.load(os.path.join(golden_dir, "turn_samples.npz"))
    names = [k for k in z.files if k.endswith("_records")]
    assert len(names) == 4
    for name in names:
        recs = z[name]
        path = str(tmp_path / (name + ".bin"))
        api.write_samples_file(path, recs)
        assert open(path, "rb").read() == np.uint64(len(recs)).tobytes() + recs.tobytes(), name


@pytest.mark.gpu
def test_device_recording_matches_oracle_replay():
    """az_selfplay_run with recording: every finished game's samples (state image, policy target, outcome) equal an oracle replay"""
    from alphazero_risk_b200 import api
    if api.lib().az_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu suite must run on a B200")
    n, moves, sims = 12, 900, 4
    env = api.Env(n, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1), first_game_id=3)
    env.reset(SEED)
    mc = api.Mcts(env, evaluator=api.EVAL_PSEUDO)
    mc.record(capacity_samples=n * moves, max_moves_per_game=1024)
    mc.selfplay(moves)
    recs, dropped = mc.samples()
    assert dropped == 0 and mc.counters()["errors"] == 0
    # oracle replay: the expected records of every game that finished, grouped per game
    rules = po.default_rules(mcts_simulations=sims, threads_per_mcts=1)
    expected = []
    for g in range(n):
        o, t = po.OracleGame(rules), po.OracleMcts(rules, "pseudo")
        o.new_game(SEED, 3 + g, 0)
        cur = []
        for ply in range(moves):
            a = t.search(o, SEED, 3 + g, ply)
            cur.append((po.RoState.from_buffer_copy(o.s), a["pi"].copy()))
            mv = t.pick(a["pi"], o.s.round <= rules.temperature_threshold, SEED, 3 + g, ply)
            assert o.move(mv, SEED, 3 + g, ply) == 0
            st = o.status()
            if st != -1:
                game = []
                for s, pi in cur:
                    o2 = po.OracleGame(rules); o2.s = s
                    game.append(o2.sample_record(pi, st))
                expected.append(np.stack(game).tobytes())
                cur = []
                o.new_game(SEED, 3 + g, ply + 1)
                t.clear()
    assert len(expected) >= n // 2, "too few finished games for a meaningful check"
    assert sum(len(e) for e in expected) == recs.size
    # games finish in a data-dependent order; each game's records are contiguous in the queue
    blob, left, pos = recs.tobytes(), sorted(expected, key=len, reverse=True), 0
    while pos < len(blob):
        hit = [e for e in left if blob.startswith(e, pos)]
        assert hit, "record stream at byte %d matches no expected game" % pos
        left.remove(hit[0]); pos += len(hit[0])
    assert not left
    # a second drain is empty; the staged samples of the running games are untouched
    again, _ = mc.samples()
    assert len(again) == 0
    mc.close(); env.close()


@NEED_REF
@pytest.mark.parametrize("rule_kw", [{}, {"min_unit_move": 1, "allow_yield": 0, "max_game_rounds": 40}], ids=["default_rules", "unit_move_1_no_yield"])
@pytest.mark.parametrize("pairing", ["script_vs_script", "script_vs_random"])
def test_scripted_turn_samples_match_reference(pairing, rule_kw, tmp_path):
    """Player::addTrainingSample inside ScriptPlayer / RandomPlayer turns (script_player.cpp:105-198, random_player.cpp:29-82) and
    the values gameFinished -> updateValues gives them: real reference players with ONE shared NNTrainDataStorage, as
    AlphaZeroTrainer::trainOnGeneratedData sets them up (alphazero_trainer.cpp:242-268), against ro_*_turn_rec; compared on the bytes
    saveTrainingSamples writes (NNInputData padding bytes excluded)"""
    L = po.ref_lib()
    rules = po.default_rules(**rule_kw)
    po.ref_apply_rules(rules)
    keep = np.ones(265, bool); keep[[1 + 43, 1 + 46, 1 + 47]] = False
    total, skips = 0, 0
    for g in range(6):
        ref, orc = po.RefGame(), po.OracleGame(rules)
        ref.new_game(SEED, 500 + g, 0); orc.new_game(SEED, 500 + g, 0)
        st = L.ref_storage_new()
        rs, os_ = [L.ref_script_new(), L.ref_script_new()], [po.new_script(), po.new_script()]
        rr = L.ref_random_new(1)
        for h in rs:
            L.ref_script_set_storage(h, st)
        L.ref_random_set_storage(rr, st)
        sink = po.TurnSink(1 << 15)
        ply = 0
        while ref.status() == -1:
            cur = orc.s.cur
            if pairing == "script_vs_script" or cur == 0:
                assert ref.script_turn(rs[cur], SEED, 500 + g, ply) == 0, L.ref_last_error()
                assert orc.script_turn_rec(os_[cur], SEED, 500 + g, ply, sink) == 0
            else:
                assert ref.random_turn(rr, SEED, 500 + g, ply) == 0, L.ref_last_error()
                assert orc.random_turn_rec(SEED, 500 + g, ply, sink) == 0
            ply += 1
            assert L.ref_storage_count(st) == len(sink), "game %d ply %d" % (g, ply)
        status = ref.status()
        assert status == orc.status()
        L.ref_script_game_finished(rs[0], status, int(orc.s.round))      # Game::playGame end: every player's gameFinished
        if pairing == "script_vs_script":
            L.ref_script_game_finished(rs[1], status, int(orc.s.round))
        else:
            L.ref_random_game_finished(rr, status, int(orc.s.round))
        path = str(tmp_path / ("g%d.bin" % g))
        assert L.ref_storage_save(st, path.encode()) == 0
        raw = np.fromfile(path, np.uint8)
        n = int(raw[:8].view(np.uint64)[0])
        assert n == len(sink) and raw.size == 8 + 265 * n
        theirs, ours = raw[8:].reshape(n, 265), sink.records(status, orc)
        assert (theirs[:, keep] == ours[:, keep]).all()
        total += n
        skips += int((sink.moves[:n] == po.SKIP).sum())
        for h in rs:
            L.ref_script_free(h)
        L.ref_random_free(rr); L.ref_storage_free(st)
    po.ref_apply_rules(po.default_rules())                  # the reference's SETTINGS are process-wide
    assert total > 1500 and (skips > 0 or pairing == "script_vs_script")     # the script's fortify rarely has nothing to move


def _well_formed(recs):
    """every record is a written one: player 0/1, the mirrored playerIndex inside NNInputData, 42 land bytes with army 1..32 and
    owner 0..2, value target in {-1, 0, +1}, a policy that sums to one"""
    assert recs.shape[1] == 265
    assert (recs[:, 0] <= 1).all() and (recs[:, 1 + 42] == recs[:, 0]).all()
    land = recs[:, 1:43]
    assert ((land & 63) >= 1).all() and ((land & 63) <= 32).all() and ((land >> 6) <= 2).all()
    value = recs[:, 89:93].copy().view(np.float32).reshape(-1)
    assert np.isin(value, [-1.0, 0.0, 1.0]).all()
    pol = recs[:, 93:265].copy().view(np.float32).reshape(-1, 43)
    assert (pol >= 0).all() and np.abs(pol.sum(1) - 1).max() < 1e-5


@pytest.mark.gpu
def test_output_queue_overflow_returns_only_written_records():
    """a sample queue smaller than what finishes: games that do not fit are dropped WHOLE and counted, the reservation never moves
    past the capacity, so every record a drain returns was written (no hole of stale bytes), and returned + dropped = everything
    the finished games produced.  Both recorders: the self-play one (az_selfplay_samples) and the scripted / random turn one
    (az_env_turn_samples)."""
    from alphazero_risk_b200 import api
    if api.lib().az_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu suite must run on a B200")
    n, moves, sims = 48, 700, 2
    rules = api.default_rules(mcts_simulations=sims, threads_per_mcts=1)

    def run(capacity):
        env = api.Env(n, rules=rules, first_game_id=40)
        env.reset(SEED)
        mc = api.Mcts(env, evaluator=api.EVAL_PSEUDO)
        mc.record(capacity_samples=capacity, max_moves_per_game=1024)
        mc.selfplay(moves)
        recs, dropped = mc.samples()
        again, dropped2 = mc.samples()
        assert len(again) == 0 and dropped2 == 0          # an empty drain reports nothing twice
        mc.close(); env.close()
        return recs.copy(), dropped

    full, d0 = run(n * moves)
    assert d0 == 0 and len(full) > 3000
    cap = 1000
    part, d1 = run(cap)
    assert 0 < len(part) <= cap and d1 > 0
    assert len(part) + d1 == len(full)
    _well_formed(part)
    # each returned game is one of the games of the unconstrained run, byte for byte
    fb = full.tobytes()
    assert all(fb.find(part[i].tobytes()) >= 0 for i in range(0, len(part), 37))
    # scripted / random turn recorder
    env = api.Env(64, first_game_id=9)
    env.record_turns(capacity_samples=1500, max_samples_per_game=4096)
    env.reset(SEED)
    script = np.full((64, 2), api.SCRIPT_INIT, np.uint32)
    for _ in range(400):
        if (env.play_turn(api.OPPONENT_SCRIPT, api.OPPONENT_RANDOM, script) != -1).all():
            break
    recs, dropped = env.turn_samples()
    assert 0 < len(recs) <= 1500 and dropped > 0
    _well_formed(recs)
    recs2, dropped2 = env.turn_samples()
    assert len(recs2) == 0 and dropped2 == 0
    env.close()
