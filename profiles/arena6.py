"""What a six-player arena match costs at configs[3]'s shape, next to self-play on the same slots.  Prints one JSON line.

    python profiles/arena6.py [--slots 16384] [--sims 16] [--max-game-rounds 20] [--blocks 5] [--selfplay-moves 40] [--out FILE]

Three runs in one process, on 16384 slots with bf16 networks of `blocks` residual blocks and random-init weights:
1. az_selfplay6_run: `selfplay-moves` moves of every game (after one warm-up move), timed with CUDA events;
2. an arena with ONE searcher in all six seats (seat_agent {0,0,0,0,0,0}): what the arena adds to the same searches;
3. searcher A vs searcher B (two networks of different seeds), seat_agent {0,1,1,1,1,1}: two compacted leaf batches per tick.
The matches use seat rotation and play the largest multiple of 6 games that fits the slots (16380), every game to its end; they are
timed with a host clock around Arena6.play, which ends in a device synchronise, after a warm-up match of one rotation group.
`max_game_rounds` bounds the games' length (rounds are counted from the set-up); both it and `sims` are recorded in the line.  Reported per run: simulations per second, wall time, ticks, and the tail = the fraction of ticks at which fewer than half
the slots still held a game.  The device name and power limit are read in the same run.  Writes nothing to the tree unless --out
names a file there."""
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


def match(api, env, agents, seat_agent, n_games, seed, slots):
    ar = api.Arena6(env, agents, seat_agent)
    ar.play(6, seed + 1, first_game=0)                       # warm-up: one rotation group
    t0 = time.perf_counter()
    r = ar.play(n_games, seed)
    dt = time.perf_counter() - t0
    active = ar.active_slots()
    ar.close()
    plies = r["plies"].astype(np.int64)
    return dict(wall_s=dt, sims=r["sims"], sims_per_sec=r["sims"] / dt, evals=r["evals"], ticks=r["ticks"],
                tail_frac=float((active < slots / 2).mean()), ticks_below_half=int((active < slots / 2).sum()),
                games=r["count"], draws=r["draw"], win=r["win"], win_seat=r["win_seat"], moves=r["moves"], errors=r["errors"],
                plies=dict(min=int(plies.min()), median=float(np.median(plies)), mean=float(plies.mean()), max=int(plies.max())))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slots", type=int, default=16384)
    ap.add_argument("--sims", type=int, default=16)
    ap.add_argument("--max-game-rounds", type=int, default=20)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--selfplay-moves", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from alphazero_risk_b200 import api
    if not torch.cuda.is_available() or api.lib().az_device_count() == 0:
        sys.exit("no CUDA device: this measurement needs the GPU")
    seed = 0x5EED0006
    dev = device_info(torch)
    stream = torch.cuda.current_stream()
    rules = api.default_rules(mcts_simulations=args.sims, threads_per_mcts=1, max_game_rounds=args.max_game_rounds)
    na, nb = api.Net(blocks=args.blocks, seed=1234), api.Net(blocks=args.blocks, seed=4321)
    na.finalize(); nb.finalize()
    n_games = args.slots - args.slots % 6
    env = api.Env6(args.slots, rules=rules)
    ma = api.Mcts6(env, net=na, evaluator=api.EVAL_NN, precision=api.BF16)
    mb = api.Mcts6(env, net=nb, evaluator=api.EVAL_NN, precision=api.BF16)
    # 1. self-play on the same slots (default stream, as the matches)
    env.reset(seed)
    ma.selfplay(1)
    torch.cuda.synchronize()
    ma.counters(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    ma.selfplay(args.selfplay_moves)
    e1.record(stream)
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    cnt = ma.counters()
    selfplay = dict(moves=args.selfplay_moves, wall_s=ms * 1e-3, sims=cnt["sims"], sims_per_sec=cnt["sims"] / (ms * 1e-3),
                    games_ended=cnt["games"], errors=cnt["errors"])
    print("selfplay6:", json.dumps(selfplay), file=sys.stderr, flush=True)
    # 2. one searcher in every seat; 3. A vs B
    solo = match(api, env, [ma], (0, 0, 0, 0, 0, 0), n_games, seed, args.slots)
    print("arena_one_searcher:", json.dumps(solo), file=sys.stderr, flush=True)
    versus = match(api, env, [ma, mb], (0, 1, 1, 1, 1, 1), n_games, seed, args.slots)
    ma.close(); mb.close(); env.close(); na.close(); nb.close()
    line = dict(metric="arena6", device=dev,
                config=dict(slots=args.slots, games=n_games, sims=args.sims, max_game_rounds=args.max_game_rounds, blocks=args.blocks,
                            precision="bf16", weights="random init (seeds 1234 / 4321)", rotate_seats=True, seed=seed,
                            timing="selfplay: CUDA events; matches: host clock around Arena6.play (ends in a device synchronise)"),
                selfplay6=selfplay, arena_one_searcher=solo, arena_a_vs_b=versus,
                arena_over_selfplay_sims_per_sec=dict(one_searcher=solo["sims_per_sec"] / selfplay["sims_per_sec"],
                                                      a_vs_b=versus["sims_per_sec"] / selfplay["sims_per_sec"]))
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if solo["errors"] or versus["errors"] or selfplay["errors"]:
        sys.exit("search overflow counters are not zero")


if __name__ == "__main__":
    main()
