"""What generated six-player games (az_env6_play, SIXPLAYER.md §6) cost, and what a first network trained on them does.  Prints one
JSON line.

    python profiles/generated6.py [--slots 16384] [--plies 2000] [--repeats 5] [--train-records 2000000] [--epochs 3]
                                  [--sims 200] [--max-game-rounds 20] [--blocks 5] [--skip-matches] [--out FILE]

1. Generation rate on `slots` games: six variants alternated in one process, `repeats` times each, every timed call starting from a
   fresh deal (reset) with the same seed and playing `plies` plies.  On an env without recording: az_env6_rollout; play with six
   random seats (which launches k_env6_rollout itself); six scripts (k_env6_play<false>).  On an env with recording enabled
   (k_env6_play<true>): six random seats with record_seats = 0 (k_env6_play's own random player, nothing recorded); six scripts,
   every seat recorded; one script (seat 0) + five random seats, seat 0 recorded.  Kernel time
   from the env's CUDA events (az_env6_last_kernel_ms); plies/s = slots x plies / kernel time; records/s = records queued by the
   call / kernel time.  A warm-up call of every variant comes first.
2. The first trained six-player network: `train_records` records of six-script games (every seat recorded, max_game_rounds as the
   match below) train a bf16 network of `blocks` residual blocks (13 planes, one value output, random init seed 1234: the network
   shape of profiles/script6.json's match) for `epochs` epochs with az_nn_train6; per-epoch losses.  Then the top-1 agreement of its
   policy (bf16 forward, restricted to the legal moves) with the script on held-out positions from fresh script games (other game
   ids).  Then script6.json's match twice: one searcher at `sims` simulations vs 5 scripts, 16380 rotated games, once with the
   trained network and once with the random-init network.
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


def rates(api, slots, plies, repeats, seed):
    S, R = api.SCRIPT6, None
    plain, rec = api.Env6(slots), api.Env6(slots)
    rec.record(capacity_samples=slots * plies, max_samples_per_game=4096)
    variants = [("rollout", plain, None, 0), ("play_random", plain, [R] * 6, 0), ("play_scripts", plain, [S] * 6, 0),
                ("play_random_recording_env", rec, [R] * 6, 0), ("play_scripts_recorded", rec, [S] * 6, 0x3f),
                ("play_1script_5random_recorded", rec, [S] + [R] * 5, 0x01)]
    res = {v[0]: dict(plies_per_sec=[], records_per_sec=[], records=[], ms=[]) for v in variants}

    def once(env, kinds, seats):
        env.reset(seed)
        if kinds is None:
            env.rollout(plies)
        else:
            env.play(kinds, plies, seats)
        ms = env.last_kernel_ms()
        if env is plain:
            return ms, 0
        recs, dropped = env.samples()
        assert dropped == 0
        return ms, len(recs)

    for _, env, kinds, seats in variants:       # warm-up
        once(env, kinds, seats)
    for _ in range(repeats):
        for name, env, kinds, seats in variants:
            ms, k = once(env, kinds, seats)
            r = res[name]
            r["ms"].append(ms); r["records"].append(k)
            r["plies_per_sec"].append(slots * plies / (ms * 1e-3)); r["records_per_sec"].append(k / (ms * 1e-3))
    plain.close(); rec.close()
    out = {}
    for name, r in res.items():
        out[name] = dict(kernel_ms=spread(r["ms"]), plies_per_sec=spread(r["plies_per_sec"]), records=r["records"],
                         records_per_sec=spread(r["records_per_sec"]),
                         kernel_ms_spread_frac=(max(r["ms"]) - min(r["ms"])) / float(np.median(r["ms"])))
    base = out["rollout"]["plies_per_sec"]["median"]
    for name in out:
        out[name]["plies_per_sec_over_rollout"] = out[name]["plies_per_sec"]["median"] / base
    return out


def generate(api, rules, slots, first, want, seed):
    """records of six-script games, every seat recorded, until `want` records are queued (whole games)"""
    env = api.Env6(slots, rules=rules, first_game_id=first)
    env.reset(seed)
    env.record(capacity_samples=want + slots * 1200, max_samples_per_game=2048)
    got, total, t0 = [], 0, time.perf_counter()
    while total < want:
        env.play([api.SCRIPT6] * 6, 400, 0x3f)
        r, dropped = env.samples()
        assert dropped == 0
        got.append(r); total += len(r)
    dt = time.perf_counter() - t0
    env.close()
    return np.concatenate(got), dt


def agreement(api, net, recs, rules):
    """top-1 agreement of the network's legal-masked policy with the recorded (scripted) action"""
    n = 16384
    env = api.Env6(n, rules=rules)
    agree = total = 0
    for i in range(0, len(recs) - n + 1, n):
        r = recs[i:i + n]
        env.import_images(r[:, :108])
        x = env.encode(planes=13)
        valid, status = env.query()
        p, _ = net.forward(x, api.BF16)
        mask = ((valid[:, None] >> np.arange(43, dtype=np.uint64)) & np.uint64(1)).astype(bool)
        pick = np.where(mask, p, -1.0).argmax(1)
        agree += int((pick == r[:, 112:284].copy().view(np.float32).argmax(1)).sum())
        total += n
    env.close()
    return dict(positions=total, top1_agreement=agree / total)


def match(api, net, rules, slots, seed):
    env = api.Env6(slots, rules=rules)
    mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
    ar = api.Arena6(env, [mc, api.SCRIPT6], (0, 1, 1, 1, 1, 1))
    ar.play(6, seed + 1, first_game=0)                       # warm-up: one rotation group
    n_games = slots - slots % 6
    t0 = time.perf_counter()
    r = ar.play(n_games, seed)
    dt = time.perf_counter() - t0
    ar.close(); mc.close(); env.close()
    plies = r["plies"].astype(np.int64)
    return dict(wall_s=dt, games=r["count"], draws=r["draw"], win=r["win"][:2], win_seat=r["win_seat"], moves=r["moves"][:2],
                sims=r["sims"], sims_per_sec=r["sims"] / dt, errors=r["errors"],
                plies=dict(min=int(plies.min()), median=float(np.median(plies)), mean=float(plies.mean()), max=int(plies.max())))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slots", type=int, default=16384)
    ap.add_argument("--plies", type=int, default=2000)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--train-records", type=int, default=2000000)
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--sims", type=int, default=200)
    ap.add_argument("--max-game-rounds", type=int, default=20)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--skip-matches", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from alphazero_risk_b200 import api
    if not torch.cuda.is_available() or api.lib().az_device_count() == 0:
        sys.exit("no CUDA device: this measurement needs the GPU")
    seed = 0x5EED0006
    dev = device_info(torch)
    rate = rates(api, args.slots, args.plies, args.repeats, seed)
    print("rates:", json.dumps(rate), file=sys.stderr, flush=True)

    rules = api.default_rules(mcts_simulations=args.sims, threads_per_mcts=1, max_game_rounds=args.max_game_rounds)
    recs, gen_s = generate(api, rules, args.slots, 0, args.train_records, seed)
    held, _ = generate(api, rules, args.slots, 1 << 24, 4 * 16384, seed)      # other game ids: positions the network never saw
    train = recs[:args.train_records]
    net = api.Net(blocks=args.blocks, seed=1234)
    net.train_precision(api.BF16)
    t0 = time.perf_counter()
    lp, lv = net.train6(train, epochs=args.epochs, batch_size=512, seed=1)
    train_s = time.perf_counter() - t0
    z = train[:, 108:112].copy().view(np.float32).reshape(-1)
    trained = dict(records=len(train), games_generation_s=gen_s, value_target_mean=float(z.mean()), epochs=args.epochs, batch=512,
                   precision="bf16", train_s=train_s, epoch_loss_policy=[float(v) for v in lp], epoch_loss_value=[float(v) for v in lv],
                   held_out=agreement(api, net, held, rules))
    init = api.Net(blocks=args.blocks, seed=1234)
    trained["random_init_held_out"] = agreement(api, init, held, rules)
    print("trained:", json.dumps(trained), file=sys.stderr, flush=True)
    matches = None
    if not args.skip_matches:
        matches = dict(trained=match(api, net, rules, args.slots, seed))
        print("match trained:", json.dumps(matches["trained"]), file=sys.stderr, flush=True)
        init.finalize()
        matches["random_init"] = match(api, init, rules, args.slots, seed)
        print("match random init:", json.dumps(matches["random_init"]), file=sys.stderr, flush=True)
    net.close(); init.close()
    line = dict(metric="generated6", device=dev,
                config=dict(slots=args.slots, plies=args.plies, repeats=args.repeats, seed=seed, train_records=args.train_records,
                            blocks=args.blocks, sims=args.sims, max_game_rounds=args.max_game_rounds, seat_agent=[0, 1, 1, 1, 1, 1],
                            timing="rates: CUDA events around each az_env6_play / az_env6_rollout kernel; training and matches: host clock"),
                generation=rate, training=trained, matches=matches)
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if matches and (matches["trained"]["errors"] or matches["random_init"]["errors"]):
        sys.exit("search overflow counters are not zero")


if __name__ == "__main__":
    main()
