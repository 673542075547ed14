"""Times the two pooled rollout kernels side by side at the bench shape: k_env_rollout (land bytes copied through a lane column
every move, entry az_env_rollout_lane_columns) and k_env_rollout_slots (land bytes kept in the pool slot, az_env_rollout).

    python profiles/rollout_slots.py [--games 65536] [--lockstep 512] [--steps 20] [--warmup 3] [--repeats 5] [--out FILE]

Both kernels start every repeat from the same deal (reset, --warmup untimed launches, then --steps timed launches with a 256 MiB
L2 flush before each, as bench.py times its headline line), alternating old / new within each repeat.  Before timing, one launch of
each from the same deal must leave identical State images and counters.  Prints one JSON line (and writes it to --out)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED = 0x5EED0001


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return {"nvidia_smi": None}
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=65536)
    ap.add_argument("--lockstep", type=int, default=512)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    from alphazero_risk_b200 import api

    n, S = args.games, args.lockstep
    env = api.Env(n, device=0)
    L = env.L
    L.az_env_rollout_lane_columns.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    stream = torch.cuda.current_stream()
    sptr = stream.cuda_stream
    kernels = {
        "k_env_rollout": lambda: api.check(L.az_env_rollout_lane_columns(env.h, S, sptr)),
        "k_env_rollout_slots": lambda: api.check(L.az_env_rollout(env.h, S, sptr)),
    }

    # same results: one launch of each from the same deal
    images, counts = {}, {}
    for name, launch in kernels.items():
        env.reset(SEED, stream=sptr)
        env.counters(reset=True, stream=sptr)
        launch()
        torch.cuda.synchronize()
        images[name], counts[name] = env.export_aos(), env.counters(reset=True, stream=sptr)
    same = bool(np.array_equal(images["k_env_rollout"], images["k_env_rollout_slots"])) and \
        counts["k_env_rollout"] == counts["k_env_rollout_slots"]

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # > 126 MB L2
    ms = {name: [] for name in kernels}
    for _ in range(args.repeats):
        for name, launch in kernels.items():
            env.reset(SEED, stream=sptr)
            for _ in range(args.warmup):
                launch()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            for i in range(args.steps):
                flush.fill_(i & 0xff)
                ev[i][0].record(stream)
                launch()
                ev[i][1].record(stream)
            torch.cuda.synchronize()
            ms[name].append(sum(a.elapsed_time(b) for a, b in ev) / args.steps)
    env.close()

    res = {}
    for name, v in ms.items():
        gs = [n * S / (t * 1e-3) / 1e9 for t in v]
        res[name] = {"ms_per_launch": [round(t, 4) for t in v], "G_steps_per_s": [round(g, 3) for g in gs],
                     "median_G_steps_per_s": round(float(np.median(gs)), 3), "spread_G_steps_per_s": round(max(gs) - min(gs), 3)}
    old, new = res["k_env_rollout"], res["k_env_rollout_slots"]
    line = {"what": "pooled env rollout: land bytes through a lane column (k_env_rollout) vs kept in the slot (k_env_rollout_slots)",
            "shape": {"games": n, "moves_per_launch": S, "timed_launches": args.steps, "warmup": args.warmup, "repeats": args.repeats,
                      "l2": "256 MiB flush before every timed launch"},
            "card": card(), "same_results": same, "kernels": res,
            "speedup_median": round(new["median_G_steps_per_s"] / old["median_G_steps_per_s"], 4),
            "worst_new_over_best_old": round(min(new["G_steps_per_s"]) / max(old["G_steps_per_s"]), 4)}
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")
    if not same:
        sys.exit("the two kernels disagree")


if __name__ == "__main__":
    main()
