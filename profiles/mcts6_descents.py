"""What several descents per tree (az_rules.concurrent_descents = K, SIXPLAYER.md §2) do to six-player search throughput.  Prints one
JSON line.

    python profiles/mcts6_descents.py [--repeats 3] [--blocks 5] [--out FILE]

Three measurements in one process, bf16 networks of `blocks` residual blocks with random-init weights:
1. az_selfplay6_run at 16384 games x 200 simulations, K in {1, 2, 4};
2. az_selfplay6_run at 1024 games x 200 simulations, K in {1, 4, 8};
3. profiles/arena6.py's A-vs-B match (16380 games with seat rotation, 16 simulations, max_game_rounds 20, seat_agent {0,1,1,1,1,1},
   two networks of different seeds), K in {1, 4}: wall time, ticks and the tail = the fraction of ticks at which fewer than half the
   slots still held a game.
Every K has its own env / Mcts6 pair (K is an env rule) over the same seeded games: self-play starts from a 3000-step uniform-random
rollout and is warmed up by one move.  The K values are timed in alternation, `repeats` times each, so the spread between repeats of
one K is visible next to the difference between Ks.  Self-play is timed with CUDA events around `moves` moves; a match with a host
clock around Arena6.play (which ends in a device synchronise), after a warm-up match of one rotation group.  The device name and power
limit are read in the same run.  Writes nothing to the tree unless --out names a file there."""
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

SEED = 0x5EED0008


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


def selfplay(api, torch, net, games, sims, ks, moves, repeats):
    stream = torch.cuda.current_stream()
    pairs = {}
    for K in ks:
        env = api.Env6(games, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K))
        env.reset(SEED)
        env.rollout(3000)
        mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
        mc.selfplay(1)                                          # warm-up
        torch.cuda.synchronize()
        mc.counters(reset=True)
        pairs[K] = (env, mc)
    rates, errors = {K: [] for K in ks}, {K: 0 for K in ks}
    for _ in range(repeats):
        for K in ks:
            env, mc = pairs[K]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            mc.selfplay(moves)
            e1.record(stream)
            e1.synchronize()
            cnt = mc.counters(reset=True)
            rates[K].append(cnt["sims"] / (e0.elapsed_time(e1) * 1e-3))
            errors[K] += cnt["errors"]
    for env, mc in pairs.values():
        mc.close(); env.close()
    out = {str(K): dict(sims_per_sec=spread(rates[K]), errors=errors[K]) for K in ks}
    base = np.median(rates[ks[0]])
    for K in ks:
        out[str(K)]["over_k1_median"] = float(np.median(rates[K]) / base)
    return dict(games=games, sims=sims, moves_per_run=moves, by_k=out)


def arena(api, na, nb, slots, sims, rounds, ks, repeats):
    n_games = slots - slots % 6
    setups = {}
    for K in ks:
        env = api.Env6(slots, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, max_game_rounds=rounds,
                                                      concurrent_descents=K))
        ma = api.Mcts6(env, net=na, evaluator=api.EVAL_NN, precision=api.BF16)
        mb = api.Mcts6(env, net=nb, evaluator=api.EVAL_NN, precision=api.BF16)
        ar = api.Arena6(env, [ma, mb], (0, 1, 1, 1, 1, 1))
        ar.play(6, SEED + 1, first_game=0)                      # warm-up: one rotation group
        setups[K] = (env, ma, mb, ar)
    runs = {K: [] for K in ks}
    for _ in range(repeats):
        for K in ks:
            ar = setups[K][3]
            t0 = time.perf_counter()
            r = ar.play(n_games, SEED)
            dt = time.perf_counter() - t0
            active = ar.active_slots()
            runs[K].append(dict(wall_s=dt, ticks=r["ticks"], tail_frac=float((active < slots / 2).mean()), sims=r["sims"],
                                sims_per_sec=r["sims"] / dt, evals=r["evals"], errors=r["errors"], draws=r["draw"], win=r["win"],
                                plies_mean=float(r["plies"].astype(np.int64).mean())))
    for env, ma, mb, ar in setups.values():
        ar.close(); ma.close(); mb.close(); env.close()
    out = {}
    for K in ks:
        out[str(K)] = dict(wall_s=spread([x["wall_s"] for x in runs[K]]), sims_per_sec=spread([x["sims_per_sec"] for x in runs[K]]),
                           ticks=runs[K][0]["ticks"], tail_frac=runs[K][0]["tail_frac"], runs=runs[K])
        out[str(K)]["wall_over_k1_median"] = out[str(K)]["wall_s"]["median"] / float(np.median([x["wall_s"] for x in runs[ks[0]]]))
    return dict(slots=slots, games=n_games, sims=sims, max_game_rounds=rounds, seat_agent=[0, 1, 1, 1, 1, 1], by_k=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--arena-repeats", type=int, default=2)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--big-moves", type=int, default=2, help="self-play moves per timed run at 16384 games")
    ap.add_argument("--small-moves", type=int, default=8, help="self-play moves per timed run at 1024 games")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from alphazero_risk_b200 import api
    if not torch.cuda.is_available() or api.lib().az_device_count() == 0:
        sys.exit("no CUDA device: this measurement needs the GPU")
    dev = device_info(torch)
    na, nb = api.Net(blocks=args.blocks, seed=1234), api.Net(blocks=args.blocks, seed=4321)
    na.finalize(); nb.finalize()
    big = selfplay(api, torch, na, 16384, 200, [1, 2, 4], args.big_moves, args.repeats)
    print("selfplay 16384:", json.dumps(big), file=sys.stderr, flush=True)
    small = selfplay(api, torch, na, 1024, 200, [1, 4, 8], args.small_moves, args.repeats)
    print("selfplay 1024:", json.dumps(small), file=sys.stderr, flush=True)
    match = arena(api, na, nb, 16384, 16, 20, [1, 4], args.arena_repeats)
    na.close(); nb.close()
    line = dict(metric="mcts6_descents", device=dev,
                config=dict(blocks=args.blocks, precision="bf16", weights="random init (seeds 1234 / 4321)", seed=SEED,
                            repeats=args.repeats, arena_repeats=args.arena_repeats,
                            timing="self-play: CUDA events; matches: host clock around Arena6.play (ends in a device synchronise)"),
                selfplay_16384=big, selfplay_1024=small, arena_a_vs_b=match)
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    errs = [v["errors"] for s in (big, small) for v in s["by_k"].values()] + \
           [x["errors"] for v in match["by_k"].values() for x in v["runs"]]
    if any(errs):
        sys.exit("search overflow counters are not zero")


if __name__ == "__main__":
    main()
