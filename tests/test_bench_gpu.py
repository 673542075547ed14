"""GPU suite: bench.py --dump-outputs writes what the timed rollouts computed, the same arrays on every run with the same arguments,
and --steps sets the number of timed rollout launches."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0x5EED0001
GAMES, LOCKSTEP, WARMUP = 4096, 64, 3
SMALL = ["--games", str(GAMES), "--lockstep", str(LOCKSTEP), "--warmup", str(WARMUP), "--no-selfplay", "--play-games", "0",
         "--train-batch", "0", "--env6-games", "0", "--no-cpu-baseline", "--e2e-shards", "2"]


def bench(steps, out):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--dump-outputs", str(out)] + SMALL,
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return json.loads(p.stdout)


def test_dump_outputs_repeat_and_follow_the_timed_steps(tmp_path):
    steps = 2
    line = bench(steps, tmp_path / "a")
    bench(steps, tmp_path / "b")
    assert line["steps"] == steps
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b")) == ["counters.npy", "game_ids.npy", "state_images.npy"]
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and a.shape == b.shape and (a == b).all(), f
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    cnt = np.load(tmp_path / "a" / "counters.npy")
    assert cnt[0] == GAMES * LOCKSTEP * steps and cnt[1] == cnt[2] + cnt[3] + cnt[4] and cnt[1] > 0
    # the dumped images are the games dealt from the seed after the warm-up and the timed launches, replayed on the oracle
    img = np.load(tmp_path / "a" / "state_images.npy")
    ids = np.load(tmp_path / "a" / "game_ids.npy")
    assert img.shape == (GAMES, 160) and (ids == np.arange(GAMES)).all()
    o = po.OracleGame()
    for g in range(0, GAMES, 257):
        o.new_game(SEED, g, 0)
        ply = 0
        for _ in range(LOCKSTEP * (WARMUP + steps)):
            if o.status() != -1:
                o.new_game(SEED, g, ply)
            assert o.move(o.random_action(SEED, g, ply), SEED, g, ply) == 0
            ply += 1
        assert (img[g].astype(np.uint8) == o.data()).all(), g
