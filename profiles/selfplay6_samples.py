"""What six-player sample recording and six-player training cost, at configs[3]'s shape.  Prints one JSON line.

    python profiles/selfplay6_samples.py [--games 16384] [--sims 200] [--blocks 5] [--moves 2] [--rounds 4] [--train-records 32768]

1. Self-play: two identical env6 / Mcts6 pairs (same seed, 16384 games x 200 simulations, bf16 network with random-init weights),
   one recording (Mcts6.record, default staging of 4096 moves per game), one not.  They are timed in alternation, `moves` moves per
   turn, `rounds` turns each, with CUDA events.  The games start from a 3000-step uniform-random rollout, so some of them end inside
   the timed window and their records are written there.  Both pairs must end with the same game images and counters: recording
   changes nothing the search computes.
2. Training: az_nn_train (265-byte two-player records) and az_nn_train6 (288-byte six-player records) in bf16 training mode, batch 512,
   timed in alternation on two networks with the same initial weights.  The six-player records hold real positions (the env's images);
   the two-player records hold well-formed synthetic positions, since a training step's cost does not depend on the values.
The device name and power limit are read in the same run.  Writes nothing to the tree."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def device_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(out[0]), float(out[1])
    except Exception as e:  # noqa: BLE001 - reported, not hidden
        info["power_limit_w"] = None
        info["power_limit_error"] = repr(e)
    return info


def records2(n, rng):
    """well-formed 265-byte two-player records: player, NNInputData (lands, player, round, 10 floats), value, policy"""
    r = np.zeros((n, 265), np.uint8)
    cur = rng.integers(0, 2, n)
    r[:, 0] = cur
    r[:, 1:43] = (rng.integers(1, 33, (n, 42)) | (rng.integers(0, 3, (n, 42)) << 6)).astype(np.uint8)
    r[:, 43] = cur
    r[:, 45] = rng.integers(1, 58, n)
    f = rng.random((n, 10), dtype=np.float32)
    f[:, 3:9] = np.eye(6, dtype=np.float32)[rng.integers(0, 6, n)]
    r[:, 49:89] = f.view(np.uint8)
    r[:, 89:93] = rng.choice(np.array([-1.0, 0.0, 1.0], np.float32), n).view(np.uint8).reshape(n, 4)
    pi = rng.random((n, 43), dtype=np.float32)
    r[:, 93:] = (pi / pi.sum(1, keepdims=True)).astype(np.float32).view(np.uint8)
    return r


def records6(images, valid, rng):
    n = len(images)
    r = np.zeros((n, 288), np.uint8)
    r[:, :108] = images
    status = rng.choice(np.array([0, 1, 2, 3, 4, 5, -2]), n)
    cur = images[:, 98].astype(np.int64)
    z = np.where(status == -2, 0.0, np.where(status == cur, 1.0, np.float32(-1.0) / np.float32(5.0))).astype(np.float32)
    r[:, 108:112] = z.view(np.uint8).reshape(n, 4)
    mask = np.array([[(int(v) >> i) & 1 for i in range(43)] for v in valid], np.float32)
    pi = mask * rng.random((n, 43), dtype=np.float32)
    r[:, 112:284] = (pi / pi.sum(1, keepdims=True)).astype(np.float32).view(np.uint8)
    r[:, 284] = status.astype(np.int8).view(np.uint8)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=16384)
    ap.add_argument("--sims", type=int, default=200)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--moves", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--train-records", type=int, default=32768)
    args = ap.parse_args()
    import torch
    from alphazero_risk_b200 import api
    if not torch.cuda.is_available() or api.lib().az_device_count() == 0:
        sys.exit("no CUDA device: this measurement needs the GPU")
    seed = 0x5EED0001
    stream = torch.cuda.current_stream()
    sptr = stream.cuda_stream
    dev = device_info(torch)
    rules = api.default_rules(mcts_simulations=args.sims, threads_per_mcts=1)
    net = api.Net(blocks=args.blocks, seed=1234)
    net.finalize()
    arms = {}
    for name in ("plain", "record"):
        env = api.Env6(args.games, rules=rules)
        env.reset(seed, stream=sptr)
        env.rollout(3000, stream=sptr)
        mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
        if name == "record":
            mc.record(capacity_samples=args.games * 64)
        mc.selfplay(1, stream=sptr)                          # warm-up move
        torch.cuda.synchronize()
        mc.counters(reset=True, stream=sptr)
        arms[name] = dict(env=env, mc=mc, ms=[])
    for _ in range(args.rounds):
        for name in ("plain", "record"):
            a = arms[name]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            a["mc"].selfplay(args.moves, stream=sptr)
            e1.record(stream)
            e1.synchronize()
            a["ms"].append(e0.elapsed_time(e1))
    res = {}
    for name, a in arms.items():
        cnt = a["mc"].counters(stream=sptr)
        sims = cnt["sims"] / (args.rounds * args.moves)          # per move
        res[name] = dict(sims_per_sec=[sims / (ms * 1e-3 / args.moves) for ms in a["ms"]], ms_per_move=[ms / args.moves for ms in a["ms"]],
                         counters=cnt, image=a["env"].export(stream=sptr))
    recs, dropped = arms["record"]["mc"].samples(stream=sptr)
    same = bool((res["plain"]["image"] == res["record"]["image"]).all()) and res["plain"]["counters"] == res["record"]["counters"]
    images = res["plain"]["image"]
    valid, _ = arms["plain"]["env"].query(stream=sptr)
    for a in arms.values():
        a["mc"].close(); a["env"].close()
    # ---- training: az_nn_train vs az_nn_train6, bf16 mode, batch 512
    rng = np.random.default_rng(7)
    n = args.train_records
    pick = rng.integers(0, len(images), n)
    r6, r2 = records6(images[pick], valid[pick], rng), records2(n, rng)
    nets = {}
    for name in ("train", "train6"):
        t = api.Net(blocks=args.blocks, seed=99)
        t.train_precision(api.BF16)
        nets[name] = dict(net=t, rate=[], loss=None)
    for name, fn in (("train", "train"), ("train6", "train6")):      # warm-up epoch of each
        getattr(nets[name]["net"], fn)(r2 if name == "train" else r6, 1, 512, 0)
    for rnd in range(args.rounds):
        for name in ("train", "train6"):
            t = nets[name]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            lp, lv = getattr(t["net"], name)(r2 if name == "train" else r6, 2, 512, rnd + 1)
            dt = time.perf_counter() - t0                          # the call ends with a device synchronise
            t["rate"].append(2 * (n // 512) * 512 / dt)
            t["loss"] = [float(lp[-1]), float(lv[-1])]
    for t in nets.values():
        t["net"].close()
    net.close()
    med = lambda v: float(np.median(v))  # noqa: E731
    plain, rec = med(res["plain"]["sims_per_sec"]), med(res["record"]["sims_per_sec"])
    line = dict(metric="selfplay6_samples", device=dev,
                config=dict(games=args.games, sims=args.sims, blocks=args.blocks, precision="bf16", moves_per_turn=args.moves,
                            rounds=args.rounds, start="3000-step uniform-random rollout", max_moves_per_game=4096),
                selfplay6=dict(plain_sims_per_sec=res["plain"]["sims_per_sec"], record_sims_per_sec=res["record"]["sims_per_sec"],
                               plain_median=plain, record_median=rec, record_cost_frac=(plain - rec) / plain,
                               games_ended=res["record"]["counters"]["games"], records_written=int(len(recs)), dropped=dropped,
                               recording_invisible=same),
                train=dict(batch=512, precision="bf16", records=n, epochs_per_turn=2,
                           train_samples_per_sec=nets["train"]["rate"], train6_samples_per_sec=nets["train6"]["rate"],
                           train_median=med(nets["train"]["rate"]), train6_median=med(nets["train6"]["rate"]),
                           ratio_train6_over_train=med(nets["train6"]["rate"]) / med(nets["train"]["rate"]),
                           last_losses=dict(train=nets["train"]["loss"], train6=nets["train6"]["loss"])))
    print(json.dumps(line))
    if not same:
        sys.exit("recording changed what the search computed")


if __name__ == "__main__":
    main()
