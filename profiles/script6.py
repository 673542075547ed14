"""What six-player matches with the scripted agent (SIXPLAYER.md §5) cost at configs[3]'s shape.  Prints one JSON line.

    python profiles/script6.py [--slots 16384] [--sims 200] [--max-game-rounds 20] [--blocks 5] [--out FILE]

On `slots` slots, seat rotation, the largest multiple of 6 games that fits the slots (16380), every game to its end:
1. the script vs 5 uniform-random players (seat_agent {0,1,1,1,1,1}, default rules): wall time and plies per second — every ply is
   played inside k_arena6_advance;
2. a bf16 searcher of `blocks` residual blocks with random-init weights at `sims` simulations vs 5 scripts (seat_agent
   {0,1,1,1,1,1}; rounds bounded by `max_game_rounds`, which counts the 13 set-up rounds): wall time, plies/s, sims/s;
3. the same match again under torch.profiler (CUDA activities): k_arena6_advance's share of the GPU kernel time, in a run of its own
   so that tracing does not slow the timed run.
Matches are timed with a host clock around Arena6.play, which ends in a device synchronise, after a warm-up match of one rotation
group.  The device name and power limit are read in the same run.  Writes nothing to the tree unless --out names a file there."""
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


def match(api, env, agents, n_games, seed):
    ar = api.Arena6(env, agents, (0, 1, 1, 1, 1, 1))
    ar.play(6, seed + 1, first_game=0)                       # warm-up: one rotation group
    t0 = time.perf_counter()
    r = ar.play(n_games, seed)
    dt = time.perf_counter() - t0
    ar.close()
    plies = r["plies"].astype(np.int64)
    return dict(wall_s=dt, plies_total=int(plies.sum()), plies_per_sec=float(plies.sum()) / dt, sims=r["sims"], sims_per_sec=r["sims"] / dt,
                ticks=r["ticks"], games=r["count"], draws=r["draw"], win=r["win"][:2], moves=r["moves"][:2], errors=r["errors"],
                plies=dict(min=int(plies.min()), median=float(np.median(plies)), mean=float(plies.mean()), max=int(plies.max())))


def advance_share(torch, api, env, agents, n_games, seed):
    from torch.profiler import ProfilerActivity, profile
    ar = api.Arena6(env, agents, (0, 1, 1, 1, 1, 1))
    ar.play(6, seed + 1, first_game=0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ar.play(n_games, seed)
        torch.cuda.synchronize()
    ar.close()
    total = advance = 0.0
    launches = 0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if e.key.startswith("Memcpy") or e.key.startswith("Memset"):
            continue
        total += t
        if "k_arena6_advance" in e.key:
            advance += t
            launches += e.count
    return dict(kernel_us_total=total, k_arena6_advance_us=advance, k_arena6_advance_launches=launches,
                k_arena6_advance_share=advance / total if total else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slots", type=int, default=16384)
    ap.add_argument("--sims", type=int, default=200)
    ap.add_argument("--max-game-rounds", type=int, default=20)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from alphazero_risk_b200 import api
    if not torch.cuda.is_available() or api.lib().az_device_count() == 0:
        sys.exit("no CUDA device: this measurement needs the GPU")
    seed = 0x5EED0006
    dev = device_info(torch)
    n_games = args.slots - args.slots % 6
    env = api.Env6(args.slots)
    vs_random = match(api, env, [api.SCRIPT6, None], n_games, seed)
    env.close()
    print("script_vs_random:", json.dumps(vs_random), file=sys.stderr, flush=True)
    rules = api.default_rules(mcts_simulations=args.sims, threads_per_mcts=1, max_game_rounds=args.max_game_rounds)
    net = api.Net(blocks=args.blocks, seed=1234)
    net.finalize()
    env = api.Env6(args.slots, rules=rules)
    mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
    vs_scripts = match(api, env, [mc, api.SCRIPT6], n_games, seed)
    print("searcher_vs_scripts:", json.dumps(vs_scripts), file=sys.stderr, flush=True)
    share = advance_share(torch, api, env, [mc, api.SCRIPT6], n_games, seed)
    print("advance_share:", json.dumps(share), file=sys.stderr, flush=True)
    mc.close(); env.close(); net.close()
    line = dict(metric="script6", device=dev,
                config=dict(slots=args.slots, games=n_games, rotate_seats=True, seed=seed, seat_agent=[0, 1, 1, 1, 1, 1],
                            script_vs_random=dict(rules="default"),
                            searcher_vs_scripts=dict(sims=args.sims, max_game_rounds=args.max_game_rounds, blocks=args.blocks,
                                                     precision="bf16", weights="random init (seed 1234)"),
                            timing="host clock around Arena6.play (ends in a device synchronise); share: torch.profiler, separate run"),
                script_vs_random=vs_random, searcher_vs_scripts=vs_scripts, searcher_vs_scripts_profile=share)
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if vs_random["errors"] or vs_scripts["errors"]:
        sys.exit("search overflow counters are not zero")


if __name__ == "__main__":
    main()
