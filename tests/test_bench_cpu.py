"""CPU suite: the reference arm of bench.py (the compiled reference, or the C restatement, timed on the host cores) prints ONE JSON
line on stdout and nothing else, with the keys the bench contract names."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout[:2000]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_committed_ncu_numbers_belong_to_the_committed_kernels():
    """profiles/traffic.json records the hashes of the sources its ncu numbers were measured on; bench.py reports roofline.traffic /
    issue_roofline from it only while they match.  The committed tree must be in that state for the three hot kernels."""
    sys.path.insert(0, ROOT)
    import bench
    for kernel in ("k_env_rollout", "k_nn_conv_tc3", "k_mcts_sim"):
        d, why = bench.ncu_capture(kernel)
        assert d is not None, why
        assert os.path.exists(os.path.join(ROOT, d["capture"])), d["capture"]


def test_dump_outputs_samples_a_fixed_set_of_games_above_the_cap(tmp_path, monkeypatch):
    """--dump-outputs over DUMP_BYTES: a seeded, sorted sample of the games, the same on every call, the files within the cap"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench

    class Env:
        n = 4096

        def export_aos(self, stream=None):
            return (np.arange(self.n * 160) % 251).astype(np.uint8).reshape(self.n, 160)

    cnt = dict(steps=7, games=3, wins=[1, 1], draws=1, illegal=0)
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), Env(), cnt, None)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["counters.npy", "game_ids.npy", "state_images.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 1 << 20
    for f in files:
        assert (np.load(tmp_path / "a" / f) == np.load(tmp_path / "b" / f)).all(), f
    ids, img = np.load(tmp_path / "a" / "game_ids.npy"), np.load(tmp_path / "a" / "state_images.npy")
    assert ids.dtype == np.float64 and img.dtype == np.float32
    assert 1000 < len(ids) < Env.n and img.shape == (len(ids), 160)
    assert (np.diff(ids) > 0).all() and ids[0] >= 0 and ids[-1] < Env.n
    assert (img == Env().export_aos()[ids.astype(int)]).all()
    assert list(np.load(tmp_path / "a" / "counters.npy")) == [7, 3, 1, 1, 1, 0]
