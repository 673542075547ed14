"""What the six-player seat planes (a network with 16 input planes, SIXPLAYER.md §2) cost next to the 13-plane network.  Prints one
JSON line.

    python profiles/planes6.py [--repeats 3] [--blocks 5] [--out FILE]

Two measurements in one process, bf16 networks of `blocks` residual blocks with six value outputs and random-init weights, one with 13
input planes and one with 16:
1. az_selfplay6_run at 16384 games x 200 simulations (K = 1), one env / Mcts6 pair per network over the same seeded games (a
   3000-step uniform-random rollout, then one warm-up move).  The two are timed in alternation, `repeats` times each, with CUDA events
   around `moves` moves, so the spread between repeats of one network is visible next to the difference between the networks.  The
   16-plane network's search encodes its leaves with the seat planes (504 more bytes of fp32 input per leaf) and its stem reads 16
   channels;
2. az_nn_train6 samples/s at batch 512 in bf16 training mode on the same records for both networks (records built from the
   rolled-out positions with random policy targets and final statuses), one warm-up epoch, then `repeats` timed epochs each in
   alternation (host clock; az_nn_train6 ends in a device synchronise).
The device name and power limit are read in the same run.  Writes nothing to the tree unless --out names a file there."""
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

SEED = 0x5EED0016


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


def spread(xs):
    return dict(runs=xs, median=float(np.median(xs)), min=float(min(xs)), max=float(max(xs)))


def selfplay(api, torch, nets, games, sims, moves, repeats):
    stream = torch.cuda.current_stream()
    pairs = {}
    for p, net in nets.items():
        env = api.Env6(games, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1))
        env.reset(SEED)
        env.rollout(3000)
        mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
        mc.selfplay(1)                                          # warm-up
        torch.cuda.synchronize()
        mc.counters(reset=True)
        pairs[p] = (env, mc)
    rates, errors = {p: [] for p in nets}, {p: 0 for p in nets}
    for _ in range(repeats):
        for p in nets:
            env, mc = pairs[p]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            mc.selfplay(moves)
            e1.record(stream)
            e1.synchronize()
            cnt = mc.counters(reset=True)
            rates[p].append(cnt["sims"] / (e0.elapsed_time(e1) * 1e-3))
            errors[p] += cnt["errors"]
    for env, mc in pairs.values():
        mc.close(); env.close()
    out = {str(p): dict(sims_per_sec=spread(rates[p]), errors=errors[p]) for p in nets}
    out["16"]["over_13_median"] = float(np.median(rates[16]) / np.median(rates[13]))
    return dict(games=games, sims=sims, moves_per_run=moves, by_input_planes=out)


def records(api, n, rng):
    """n six-player records (include/az_b200.h AZ_SAMPLE6_BYTES): rolled-out positions, random pi and final status"""
    env = api.Env6(n)
    env.reset(SEED + 1)
    env.rollout(500)
    img = env.export()
    env.close()
    rec = np.zeros((n, api.SAMPLE6_BYTES), np.uint8)
    rec[:, :108] = img
    status = rng.choice(np.array([0, 1, 2, 3, 4, 5, -2], np.int8), n)
    value = np.where(status == -2, 0.0, np.where(status == img[:, 98].astype(np.int8), 1.0, np.float32(-1.0) / np.float32(5.0)))
    rec[:, 108:112] = value.astype(np.float32).view(np.uint8).reshape(n, 4)
    pi = rng.random((n, 43)).astype(np.float32)
    pi /= pi.sum(1, keepdims=True)
    rec[:, 112:284] = pi.view(np.uint8).reshape(n, 172)
    rec[:, 284] = status.view(np.uint8)
    return rec


def train(api, nets, recs, batch, repeats):
    for net in nets.values():
        net.train_precision(api.BF16)
        net.train6(recs, 1, batch, 1)                          # warm-up epoch
    rates = {p: [] for p in nets}
    batches = len(recs) // batch
    for r in range(repeats):
        for p, net in nets.items():
            t0 = time.perf_counter()
            net.train6(recs, 1, batch, 2 + r)
            rates[p].append(batches * batch / (time.perf_counter() - t0))
    out = {str(p): dict(samples_per_sec=spread(rates[p])) for p in nets}
    out["16"]["over_13_median"] = float(np.median(rates[16]) / np.median(rates[13]))
    return dict(records=len(recs), batch=batch, batches_per_epoch=batches, precision="bf16", by_input_planes=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--moves", type=int, default=2, help="self-play moves per timed run at 16384 games")
    ap.add_argument("--train-records", type=int, default=65536)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from alphazero_risk_b200 import api
    if not torch.cuda.is_available() or api.lib().az_device_count() == 0:
        sys.exit("no CUDA device: this measurement needs the GPU")
    dev = device_info(torch)
    nets = {p: api.Net(blocks=args.blocks, seed=1234, value_outputs=6, input_planes=p) for p in (13, 16)}
    for net in nets.values():
        net.finalize()
    sp = selfplay(api, torch, nets, 16384, 200, args.moves, args.repeats)
    print("selfplay 16384:", json.dumps(sp), file=sys.stderr, flush=True)
    tr = train(api, nets, records(api, args.train_records, np.random.default_rng(7)), 512, args.repeats)
    for net in nets.values():
        net.close()
    line = dict(metric="planes6", device=dev,
                config=dict(blocks=args.blocks, value_outputs=6, precision="bf16", weights="random init (seed 1234)", seed=SEED, repeats=args.repeats,
                            timing="self-play: CUDA events; az_nn_train6: host clock around one epoch (ends in a device synchronise)"),
                selfplay_16384=sp, train6=tr)
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if any(v["errors"] for v in sp["by_input_planes"].values()):
        sys.exit("search overflow counters are not zero")


if __name__ == "__main__":
    main()
