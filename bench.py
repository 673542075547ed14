#!/usr/bin/env python
"""bench.py — headline benchmark of the self-play hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): raw env throughput, 65536 lockstep 2-player games per
GPU, uniform-random legal moves, finished games re-dealt in place.  One bench "step" = one
az_env_rollout launch advancing every game by --lockstep moves.  Games shard over ranks by
contiguous global id with no data-path collective (weak scaling: per-GPU work is fixed);
NCCL is used only for the barrier and the max-over-ranks reduction of the timings.

Prints ONE JSON line (rank 0).  `value` = env steps/s with the state resident in HBM;
`e2e` = the same metric through the host-buffer C-ABI calls (import 160-byte State images
from pinned host memory -> rollout -> export images + counters, copies inside the timed
region); `roofline` is for the rollout kernel; `cpu_baseline` = the reference's own CPU code
(oracle/_ref) on the box's host cores, rank 0 / N=1 only.  --impl reference times that CPU
path alone.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the tree may be read-only: the benchmark writes nothing into it

ENV_BYTES_PER_STEP = 330      # SURVEY.md §8d: 2 x 160 B State image + 8 B mask + 1 B action + 1 B status
SEED = 0x5EED0001


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1392.5))), "measured"
    return 6650.0, 1400.0, "fallback"


def ncu_capture(kernel):
    """the committed ncu --set full numbers of `kernel` (profiles/traffic.json, tools/traffic_from_ncu.py) — only if they were
    measured on the sources this library was built from; otherwise None and a reason (a capture of another binary is not evidence)"""
    import hashlib
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        d = json.load(open(p)).get(kernel)
    except (OSError, ValueError):
        return None, "profiles/traffic.json missing or unreadable"
    if d is None:
        return None, "no capture of %s in profiles/traffic.json" % kernel
    for f, want in (d.get("sources") or {"<none>": ""}).items():
        path = os.path.join(ROOT, "include" if f.endswith(".h") and not f.startswith("az_tables") else "alphazero_risk_b200/csrc", f)
        try:
            have = hashlib.sha256(open(path, "rb").read()).hexdigest()[:16]
        except OSError:
            have = None
        if have != want:
            return None, "capture %s was taken on a different %s (re-run tools/round_profile.sh)" % (d.get("capture"), f)
    return d, None


def ncu_traffic(kernel):
    """roofline.traffic (DRAM bytes per launch, ncu) plus where it comes from; null + the reason when the capture is stale"""
    d, why = ncu_capture(kernel)
    if d is None:
        sys.stderr.write("bench.py: roofline.traffic of %s not reported: %s\n" % (kernel, why))
        return {"traffic": None, "traffic_stale": why}
    return {"traffic": float(d["dram_bytes_read"]) + float(d["dram_bytes_write"]), "traffic_capture": d.get("capture")}


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons of one GPU during the timed region"""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_env_baseline(seconds_target):
    """reference CPU path for config 2 on all host threads: oracle/_ref when built, else the C port"""
    import ctypes as C
    from oracle import pyoracle as po          # the one place bench.py may execute oracle/
    threads = host_threads()
    if po.ref_available():
        L = po.ref_lib()
        po.ref_apply_rules(po.default_rules())
        out = po.BenchOut()
        L.ref_bench_env(threads, 200_000, 1, C.byref(out))              # calibrate
        rate = out.steps / max(out.seconds, 1e-9) / threads
        per_thread = int(max(200_000, rate * seconds_target))
        L.ref_bench_env(threads, per_thread, 2, C.byref(out))
        return dict(value=out.steps / out.seconds, unit="steps/s", cores=threads, kind="reference",
                    sample="%d threads x %d random-play env steps through the compiled reference "
                           "(State/UtilityNN, g++ -O3, its own std RNG), %.1f s" % (threads, per_thread, out.seconds)), out
    L = po.oracle_lib()
    out = po.BenchOut()
    L.ro_bench_env(2_000_000, SEED, C.byref(out))
    n = int(max(2_000_000, out.steps / out.seconds * seconds_target))
    L.ro_bench_env(n, SEED, C.byref(out))
    return dict(value=out.steps / out.seconds, unit="steps/s", cores=1, kind="port",
                sample="1 thread x %d random-play env steps through oracle/risk_oracle.c, %.1f s" % (n, out.seconds)), out


def cpu_selfplay_baseline(sims, seconds_target):
    """reference MCTS + env on all host threads with a NULL evaluator (uniform prior, value 0): tree + env cost only.
    TensorFlow is not installable, so the network is left out of this baseline and that is stated."""
    import ctypes as C
    from oracle import pyoracle as po
    threads = host_threads()
    if not po.ref_available():
        return {"value": None, "unit": "sims/s", "cores": 0, "kind": "port", "sample": "oracle/_ref not built"}
    L = po.ref_lib()
    po.ref_apply_rules(po.default_rules(mcts_simulations=sims, threads_per_mcts=1))
    out = po.BenchOut()
    L.ref_bench_selfplay(threads, 20, 1, None, None, C.byref(out))
    per_thread = int(max(20, out.moves / max(out.seconds, 1e-9) / threads * seconds_target))
    L.ref_bench_selfplay(threads, per_thread, 2, None, None, C.byref(out))
    po.ref_apply_rules(po.default_rules())
    res = dict(value=out.sims / out.seconds, unit="sims/s", cores=threads, kind="reference",
               sample="%d threads x %d self-play moves x %d sims through the compiled reference (AlphaZeroMCTS::simulate, T=1, "
                      "NULL evaluator: tree + env cost only, no network), %.1f s" % (threads, per_thread, sims, out.seconds))
    # the reference's network runs in TensorFlow (absent); time the PyTorch-CPU restatement of the same graph instead
    try:
        import numpy as np
        import torch
        from oracle import nn_oracle as no
        torch.set_num_threads(threads)
        rng = np.random.default_rng(0)
        shapes = {"conv/kernel": (3, 3, 13, 256), "pi/kernel": (1, 1, 256, 2), "v/kernel": (1, 1, 256, 1), "dense/kernel": (84, 43),
                  "dense/bias": (43,), "dense_1/kernel": (42, 256), "dense_1/bias": (256,), "dense_2/kernel": (256, 1), "dense_2/bias": (1,)}
        w = {}
        for name in no.variable_names(5):
            if name in shapes:
                shp = shapes[name]
            elif name.endswith("/kernel"):
                shp = (3, 3, 256, 256)
            else:
                shp = (7,) if name.startswith("conv_bn") else (2,) if name.startswith("bn_pi") else (1,) if name.startswith("bn_v") else (256,)
            w[name] = (rng.standard_normal(shp) * 0.05 + (1.0 if name.endswith(("gamma", "variance")) else 0.0)).astype(np.float32)
        x = rng.random((256, 7, 6, 13), dtype=np.float32)
        no.forward(w, x[:32], 5)
        t0 = time.perf_counter(); reps = 0
        while time.perf_counter() - t0 < 4.0:
            no.forward(w, x, 5); reps += 1
        nn_rate = reps * 256 / (time.perf_counter() - t0)
        res["nn_positions_per_sec_torch_cpu"] = nn_rate
        res["with_network_estimate_sims_per_sec"] = 1.0 / (1.0 / res["value"] + 1.0 / nn_rate)
        res["sample"] += "; 5-block network on the same cores via the PyTorch-CPU restatement (batch 256): %.0f positions/s" % nn_rate
    except Exception as e:   # noqa: BLE001
        res["nn_positions_per_sec_torch_cpu"] = None
        res["sample"] += "; torch CPU network timing failed: %s" % e
    return res


def env_config(n, S):
    """the workload both arms are measured on (BASELINE.json configs[1])"""
    return {"workload": "configs[1]: raw env throughput, %d lockstep 2-player games per GPU, uniform-random legal moves, %d moves "
                        "per launch, finished games re-dealt in place" % (n, S),
            "games_per_gpu": n, "lockstep_moves_per_step": S}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals, t0 = [], time.time()
    for i in range(args.warmup + args.steps):
        cb, out = cpu_env_baseline(1.5)
        if i >= args.warmup:
            vals.append((out.steps, out.seconds))
    steps = sum(v[0] for v in vals); secs = sum(v[1] for v in vals)
    value = steps / secs
    cb["value"] = value
    line = dict(impl="reference", metric="env_steps_per_sec", value=value, unit="steps/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * secs / max(1, args.steps), higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="u8", data="synthetic",
                config=dict(env_config(args.games, args.lockstep),
                            reference_sample="the reference's State / UtilityNN code on all host threads, one game per thread re-dealt in "
                                             "place, a bounded 1.5 s sample of the same uniform-random-move workload per step"),
                cpu_baseline=cb, e2e={"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                wall_s=time.time() - t0)
    print(json.dumps(line))


def nn_flops_per_position(blocks):
    """SURVEY.md §8d conventional count (padded taps included): 0.4981 GFLOP (5 blocks), 1.9844 GFLOP (20 blocks)"""
    return 2 * 42 * (9 * 13 * 256 + 2 * blocks * 9 * 256 * 256 + 256 * 2 + 256 * 1) + 2 * (84 * 43 + 42 * 256 + 256)


def run_selfplay(args, api, torch, dist, azd, rank, world, local, barrier, shape=None, label="configs[2]", with_tree=True):
    """BASELINE configs[2]: batched self-play, 4096 games x 64 MCTS sims/move per GPU, leaf-batched bf16
    tcgen05 network forward (5-block graph = the only GraphDef the reference ships, random-init weights).
    shape = (games, sims, blocks, moves_per_step, steps, warmup_moves) overrides the command-line shape: the cfg5 / blocks20 sub-lines."""
    from alphazero_risk_b200 import dist as azdist
    n, sims, blocks = args.sp_games, args.sp_sims, args.blocks
    moves_per_step, steps, warm_moves = args.sp_moves, max(2, min(args.steps, args.sp_steps)), None
    if shape is not None:
        n, sims, blocks, moves_per_step, steps, warm_moves = shape
    stream = torch.cuda.current_stream()
    sptr = stream.cuda_stream
    K = max(1, args.sp_descents)
    rules = api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K)
    env = api.Env(n, rules=rules, device=local, first_game_id=rank * n)
    env.reset(SEED, stream=sptr)
    net = api.Net(blocks=blocks, device=local)
    if rank == 0:
        net.init_random(1234)
    if azd is not None:       # az_dist_broadcast_weights: ncclBroadcast of rank 0's blob (replaces the checkpoint-file hand-off of
        azd.broadcast_weights([net], 0)           # alphazero_gpu_cluster.cpp:221-231)
    net.finalize()
    mc = api.Mcts(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
    if warm_moves is None:
        for _ in range(max(1, args.warmup // 2)):
            mc.selfplay(moves_per_step, stream=sptr)
    elif warm_moves > 0:
        mc.selfplay(warm_moves, stream=sptr)
    torch.cuda.synchronize()
    mc.counters(reset=True, stream=sptr)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    for i in range(steps):
        ev[i][0].record(stream)
        mc.selfplay(moves_per_step, stream=sptr)      # working set (node pools + activations) is far larger than L2
        ev[i][1].record(stream)
    barrier()
    sp_clocks = sampler.stop() if rank == 0 else None
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    cnt = mc.counters(stream=sptr)
    pool_peak, pool_cap, pool_bytes = mc.pool_stats(stream=sptr)
    # e2e: the call a host-side game loop makes per move — State images in from pinned host memory (az_env_import_aos), one
    # az_mcts_search through the host-buffer ABI (visit counts, pi, moves, status copied back), images out again; as many moves as
    # the device-timed region above
    e2e_moves = max(2, moves_per_step * steps) if shape is None else max(1, moves_per_step)
    h_img = torch.empty((n, 160), dtype=torch.uint8).pin_memory()
    env.export_aos(out=h_img.numpy(), stream=sptr)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_moves):
        env.import_aos(h_img.numpy(), stream=sptr)
        mc.search(pick_mode=api.PICK_SELFPLAY, apply_move=True, stream=sptr)
        env.export_aos(out=h_img.numpy(), stream=sptr)
    barrier()
    e2e_s = time.perf_counter() - t0
    dev_ms, e2e_ms = dev_ms, e2e_s * 1e3
    if dist is not None:
        dev_ms, e2e_ms = azdist.max_over_ranks([dev_ms, e2e_ms], dist)
        errs = cnt["errors"]                              # az_dist_gather_counters / _stats: ncclAllReduce of the tallies
        cnt = azd.gather_counters([cnt])                  # (replaces GameResults::add, game.cpp:298-309)
        cnt["errors"] = int(azd.gather_stats([[errs]])[0][0])
    tot_sims, tot_evals, tot_steps, tot_games, errors = [float(cnt[k]) for k in ("sims", "evals", "steps", "games", "errors")]
    mc.close(); net.close(); env.close()
    # ---- the tree kernels alone: the same search with the null evaluator (uniform prior, value 0: no network launches), so the
    # timed region is k_mcts_begin / k_mcts_sim / k_mcts_finish only.  HBM roofline with SURVEY §8d's per-simulation bytes.
    tree = None
    if rank == 0 and with_tree:
        env2 = api.Env(n, rules=rules, device=local, first_game_id=rank * n)
        env2.reset(SEED, stream=sptr)
        mt = api.Mcts(env2, evaluator=api.EVAL_UNIFORM)
        mt.selfplay(4, stream=sptr)
        torch.cuda.synchronize()
        mt.counters(reset=True, stream=sptr)
        t_moves = 8
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        mt.selfplay(t_moves, stream=sptr)
        b.record(stream); torch.cuda.synchronize()
        t_ms = a.elapsed_time(b)
        tc = mt.counters(stream=sptr)
        depth = tc["path_nodes"] / max(1, tc["sims"]) + 1.0           # nodes visited per simulation incl. the leaf
        bytes_per_sim = 2900.0 + 328.0 * depth
        hbm_peak, _, psrc = measured_peaks()
        tree_gbs = tc["sims"] * bytes_per_sim / (t_ms * 1e-3) / 1e9
        tree = {"sims_per_sec": tc["sims"] / (t_ms * 1e-3), "ms_per_round": t_ms / (t_moves * (sims // K + 2)), "mean_depth": depth,
                "bytes_per_sim": bytes_per_sim,
                "roofline": {"bound": "hbm", "achieved": tree_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": tree_gbs / hbm_peak,
                             **ncu_traffic("k_mcts_sim"), "peak_source": psrc,
                             "note": "null evaluator (no network): device time of the tree kernels only; algorithmic bytes per simulation = "
                                     "2.9 KB + 328 B x depth (SURVEY 8d), depth measured (path_nodes counter); one warp per game, so "
                                     "%d games give %d warps: latency-bound, not bandwidth-bound" % (n, n)},
                "errors": tc["errors"]}
        mt.close(); env2.close()
    if rank != 0:
        return None
    _, tf_peak, src = measured_peaks()
    nn_launch_positions = n * (K * (sims // K) + 1) * moves_per_step * steps  # positions pushed through the tower per rank: n per root round, n * K per simulation round
    achieved_tf = nn_launch_positions * nn_flops_per_position(blocks) / (dev_ms * 1e-3) / 1e12
    return dict(metric="mcts_sims_per_sec", value=tot_sims / (dev_ms * 1e-3), unit="sims/s", ms_per_step=dev_ms / steps, steps=steps,
                nn_evals_per_sec=tot_evals / (dev_ms * 1e-3), selfplay_env_steps_per_sec=tot_steps / (dev_ms * 1e-3),
                config={"workload": "%s: batched self-play, %d games x %d MCTS sims/move per GPU, %s, "
                                    "%d-block graph, random-init weights (seed 1234), bf16 tcgen05 forward, %d moves per step"
                                    % (label, n, sims, "T=1 semantics (one leaf per game per batch)" if K == 1 else
                                       "%d concurrent descents per tree with the active_N rule (leaf batch = %d)" % (K, n * K),
                                       blocks, moves_per_step),
                            "games_per_gpu": n, "sims_per_move": sims, "blocks": blocks, "concurrent_descents": K},
                roofline={"bound": "tensor", "achieved": achieved_tf, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved_tf / tf_peak,
                          **ncu_traffic("k_nn_conv_tc3"), "peak_source": src + " (sustained cuBLAS bf16)",
                          "executed_frac": achieved_tf * 48.0 / 42.0 / tf_peak,
                          "note": "conventional FLOPs/position (0.4981 G for 5 blocks) x positions pushed through the tower / whole-step device "
                                  "time (tree kernels, encode and heads included in the time); the 48-row board layout (42 cells + 6 zero rows per board) executes 48/42 of "
                                  "that (executed_frac); the forward runs at the board's 1 kW power cap (clocks.reasons: sw_power_cap), "
                                  "like the cuBLAS run the peak comes from; traffic = DRAM bytes of one tower-layer launch (ncu)"},
                clocks=sp_clocks,
                e2e={"value": n * sims * e2e_moves * world / (e2e_ms * 1e-3), "unit": "sims/s", "h2d_bytes_per_step": n * 160,
                     "d2h_bytes_per_step": n * (43 * 8 + 2 + 160), "steps": e2e_moves},
                gpu_launches=steps * moves_per_step * (2 + (sims // K + 1) * (1 + 1 + 1 + 2 * blocks + 1)),   # begin, finish; per round: tree, pack, stem, tower, heads
                dtype="bf16 tower / fp32 tree", results={"games_finished": tot_games, "table_errors": errors}, tree=tree,
                node_pools={"peak_nodes": pool_peak, "capacity_nodes": pool_cap, "bytes_per_game": pool_bytes,
                            "note": "rank 0; fullest pool of any game at the end of a search / nodes per pool (worst-case sizing, overflow = table_errors)"})


def run_play(args, api, torch, rank, local):
    """BASELINE configs[0] on the device: `-m play --mcts=16 --cg=1000` — AlphaZero (random-init 5-block net, bf16 tcgen05 forward,
    16 simulations per move = MCTS_SIMULATIONS 16 with the default 2 search threads, run as 2 concurrent descents per tree with the
    active_N rule) against the scripted opponent, mirror pairs.
    The reference runs 32 concurrent game threads; here every pair gets its own slot so the whole match is one lockstep batch."""
    games = args.play_games - args.play_games % 2
    slots = max(1, games // 2)
    stream = torch.cuda.current_stream(); sptr = stream.cuda_stream
    rules = api.default_rules(mcts_simulations=16, threads_per_mcts=2, concurrent_descents=2)
    env = api.Env(slots, rules=rules, device=local, first_game_id=rank * slots)
    net = api.Net(blocks=args.blocks, device=local, seed=1234)
    mc = api.Mcts(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
    arena = api.Arena(mc, api.OPPONENT_SCRIPT, mirror_games=True)
    arena.play(min(games, 2 * min(slots, 64)), SEED + 7, stream=sptr)          # warm-up match
    torch.cuda.synchronize()
    # the match is a chain of small launches with one host read-back per tick: the same match three times, the MEDIAN is reported
    ms_all = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        r = arena.play(games, SEED, stream=sptr)
        e1.record(stream); torch.cuda.synchronize()
        ms_all.append(e0.elapsed_time(e1))
    ms = sorted(ms_all)[len(ms_all) // 2]
    arena.close(); mc.close(); net.close(); env.close()
    return dict(metric="play_games_per_sec", value=r["count"] / (ms * 1e-3), unit="games/s", ms=ms, ms_runs=ms_all,
                az_sims_per_sec=r["az_sims"] / (ms * 1e-3), az_moves=r["az_moves"], opponent_turns=r["opponent_turns"],
                results={"count": r["count"], "draw": r["draw"], "win_az_script": r["win"], "win_and_started": r["win_and_started"],
                         "errors": r["errors"]},
                config={"workload": "configs[0]: -m play --mcts=16 --cg=%d, AlphaZero (random-init %d-block net, bf16) vs ScriptPlayer, both "
                                    "on the device, %d lockstep slots x 1 mirror pair, THREADS_PER_MCTS = 2 as 2 concurrent descents per tree"
                                    % (games, args.blocks, slots)})


def run_env6(args, api, torch, rank, local):
    """BASELINE configs[3]'s game: the SIX-PLAYER extension (SIXPLAYER.md; no reference semantics, checker = oracle/risk6_oracle.c).
    Environment only — 16384 lockstep six-player games, uniform-random legal moves, finished games re-dealt; the six-player search
    is specified and not built."""
    n, S = args.env6_games, args.lockstep
    stream = torch.cuda.current_stream(); sptr = stream.cuda_stream
    env = api.Env6(n, device=local, first_game_id=rank * n)
    env.reset(SEED, stream=sptr)
    for _ in range(3):
        env.rollout(S, stream=sptr)
    torch.cuda.synchronize()
    env.counters(reset=True, stream=sptr)
    steps = 5
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        ev[i][0].record(stream)
        env.rollout(S, stream=sptr)
        ev[i][1].record(stream)
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in ev) / steps
    cnt = env.counters(stream=sptr)
    env.close()
    hbm_peak, _, src = measured_peaks()
    bytes_per_step = 2 * 108 + 8 + 1 + 1                  # the 108-byte state image in and out + mask + action + status
    achieved = bytes_per_step * n * S / (ms * 1e-3) / 1e9
    return dict(metric="env6_steps_per_sec", value=n * S / (ms * 1e-3), unit="steps/s", ms_per_step=ms, steps=steps,
                config={"workload": "configs[3] game (six-player EXTENSION, SIXPLAYER.md: no reference semantics, parity unpinned; environment "
                                    "only): %d lockstep six-player games per GPU, uniform-random legal moves, %d moves per launch, finished "
                                    "games re-dealt in place" % (n, S), "games_per_gpu": n},
                roofline={"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": None,
                          "peak_source": src, "note": "algorithmic %d B/step (state image in + out, mask, action, status); like the "
                                                      "two-player rollout the kernel keeps the state on chip and is issue / latency bound; a "
                                                      "straightforward thread-per-game kernel, not tuned" % bytes_per_step},
                results={"games_finished": cnt["games"], "draws": cnt["draws"], "wins": cnt["wins"]}, gpu_launches=steps)


def run_selfplay6(args, api, torch, dist, azd, rank, world, local, barrier):
    """BASELINE configs[3] as written: six-player self-play, 16384 games x 200 simulations per move, trade-ins on — the EXTENSION of
    SIXPLAYER.md (no reference semantics, parity unpinned; checker = oracle/risk6_oracle.c).  Same tower, same bf16 tcgen05 forward;
    one move after one warm-up move."""
    from alphazero_risk_b200 import dist as azdist
    n, sims, blocks = args.cfg4_games, args.cfg4_sims, args.blocks
    stream = torch.cuda.current_stream(); sptr = stream.cuda_stream
    rules = api.default_rules(mcts_simulations=sims, threads_per_mcts=1)
    env = api.Env6(n, rules=rules, device=local, first_game_id=rank * n)
    env.reset(SEED, stream=sptr)
    env.rollout(80, stream=sptr)                          # past the 78 set-up plies: attacks, trade-ins and eliminations are live
    net = api.Net(blocks=blocks, device=local)
    if rank == 0:
        net.init_random(1234)
    if azd is not None:
        azd.broadcast_weights([net], 0)
    net.finalize()
    mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
    mc.selfplay(1, stream=sptr)
    torch.cuda.synchronize()
    mc.counters(reset=True, stream=sptr)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    mc.selfplay(1, stream=sptr)
    e1.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = e0.elapsed_time(e1)
    cnt = mc.counters(stream=sptr)
    # e2e: one az_mcts6_search through the host-buffer ABI (state images in, visit counts / pi / moves / status out)
    h_img = env.export(stream=sptr)
    barrier()
    t0 = time.perf_counter()
    env.import_images(h_img, stream=sptr)
    mc.search(pick_mode=api.PICK_SELFPLAY, apply_move=True, stream=sptr)
    env.export(stream=sptr)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    tot = [float(cnt["sims"]), float(cnt["evals"]), float(cnt["errors"])]
    if dist is not None:
        dev_ms, e2e_ms = azdist.max_over_ranks([dev_ms, e2e_ms], dist)
        tot = [float(v) for v in azd.gather_stats([[int(t) for t in tot]])[0]]
    mc.close(); net.close(); env.close()
    if rank != 0:
        return None
    _, tf_peak, src = measured_peaks()
    achieved_tf = n * (sims + 1) * nn_flops_per_position(blocks) / (dev_ms * 1e-3) / 1e12
    return dict(metric="mcts6_sims_per_sec", value=tot[0] / (dev_ms * 1e-3), unit="sims/s", ms_per_step=dev_ms, steps=1,
                nn_evals_per_sec=tot[1] / (dev_ms * 1e-3),
                config={"workload": "configs[3]: SIX-PLAYER self-play (extension, SIXPLAYER.md: no reference semantics, parity unpinned), %d games x "
                                    "%d MCTS sims/move per GPU, simple-card trade-ins, %d-block graph, random-init weights, bf16 tcgen05 forward, "
                                    "one move" % (n, sims, blocks), "games_per_gpu": n, "sims_per_move": sims, "blocks": blocks},
                roofline={"bound": "tensor", "achieved": achieved_tf, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved_tf / tf_peak,
                          **ncu_traffic("k_nn_conv_tc3"), "peak_source": src + " (sustained cuBLAS bf16)",
                          "executed_frac": achieved_tf * 48.0 / 42.0 / tf_peak,
                          "note": "as mcts.roofline; the six-player tree kernels (one warp per game, game logic on lane 0) are inside the time"},
                clocks=clocks, e2e={"value": n * sims * world / (e2e_ms * 1e-3), "unit": "sims/s", "h2d_bytes_per_step": n * 108,
                                    "d2h_bytes_per_step": n * (43 * 8 + 2 + 108), "steps": 1},
                gpu_launches=2 + (sims + 1) * (1 + 1 + 1 + 1 + 2 * blocks + 1), dtype="bf16 tower / fp32 tree", results={"table_errors": tot[2]})


def run_train(args, api, torch, local):
    """SURVEY §8f N4: one optimizer step (AlphaZeroNN::train inner loop) on a batch of SETTINGS.BATCH_SIZE = 512 synthetic samples"""
    import numpy as np
    n = args.train_batch
    rng = np.random.default_rng(5)
    net = api.Net(blocks=args.blocks, device=local, seed=1234)
    x = rng.random((n, 7, 6, 13), dtype=np.float32)
    tp = rng.random((n, 43)).astype(np.float32); tp /= tp.sum(1, keepdims=True)
    tv = rng.choice([-1.0, 0.0, 1.0], n).astype(np.float32)
    stream = torch.cuda.current_stream(); sptr = stream.cuda_stream
    flops = 3.0 * nn_flops_per_position(args.blocks) * n       # forward + data gradient + weight gradient
    out = {}
    for mode, prec in (("fp32", api.FP32), ("bf16_tcgen05", api.BF16)):
        net.train_precision(prec)
        for _ in range(2):
            net.train_step(x, tp, tv, stream=sptr)
        torch.cuda.synchronize()
        steps = 5
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            loss = net.train_step(x, tp, tv, stream=sptr)      # host batch in, two losses out, every step
        e1.record(stream); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[mode] = dict(samples_per_sec=n / (ms * 1e-3), ms_per_step=ms, achieved_tflops=flops / (ms * 1e-3) / 1e12, last_losses=list(loss))
    # AlphaZeroNN::train itself (az_nn_train: shuffled epochs over packed sample records, batches enqueued back to back): records from
    # a short device self-play with the uniform evaluator (real positions, visit-count policies, game outcomes)
    epoch = None
    try:
        env = api.Env(512, rules=api.default_rules(mcts_simulations=2, threads_per_mcts=1), device=local)
        env.reset(0x5EED0001)
        mc = api.Mcts(env, evaluator=api.EVAL_UNIFORM)
        mc.record(capacity_samples=600000, max_moves_per_game=1024)
        mc.selfplay(700)
        recs, _ = mc.samples()
        mc.close(); env.close()
        recs = recs[:(min(len(recs), 32 * n) // n) * n]
        if len(recs) >= 4 * n:
            net.train(recs, 1, n, 1)                           # warm-up epoch
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            lp, lv = net.train(recs, 2, n, 2)
            dt = time.perf_counter() - t0
            epoch = dict(samples_per_sec=2 * len(recs) / dt, ms_per_batch=dt * 1e3 / (2 * len(recs) // n), records=int(len(recs)), epochs=2,
                         losses_policy=[float(v) for v in lp], losses_value=[float(v) for v in lv],
                         note="az_nn_train wall time: record upload, per-epoch shuffle upload, every batch of every epoch, one loss read per epoch")
    except Exception as e:                                      # the step numbers above stand on their own
        epoch = dict(error=str(e))
    net.close()
    best = out["bf16_tcgen05"]
    return dict(metric="train_samples_per_sec", value=best["samples_per_sec"], unit="samples/s", ms_per_step=best["ms_per_step"], batch=n,
                blocks=args.blocks, modes=out, epoch=epoch,
                config={"workload": "one az_nn_train_step per step: batch %d, %d-block graph; value = the bf16 tcgen05 mode (the three "
                                    "contractions as tensor-core GEMMs), modes.fp32 = the fp32 parity path; host batch copied in and losses "
                                    "copied out inside the timed region" % (n, args.blocks)})


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, env, cnt, stream):
    """What the timed rollouts leave a caller: the 160-byte State image of every game (az_env_export_aos) and the counters of the
    timed steps, as float arrays (bytes and counts are exact in float32 / float64).  When the images exceed DUMP_BYTES, a fixed
    seeded sample of the games is written; game_ids.npy names the rows either way."""
    import numpy as np
    img = env.export_aos(stream=stream)
    rows = min(env.n, (DUMP_BYTES - 4096) // (img.shape[1] * 4 + 8))       # 4 KB: the three .npy headers and the counters
    ids = np.arange(env.n) if rows == env.n else np.sort(np.random.default_rng(SEED).choice(env.n, rows, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "state_images.npy"), img[ids].astype(np.float32))
    np.save(os.path.join(out_dir, "game_ids.npy"), ids.astype(np.float64))
    np.save(os.path.join(out_dir, "counters.npy"),
            np.array([cnt["steps"], cnt["games"], cnt["wins"][0], cnt["wins"][1], cnt["draws"], cnt["illegal"]], np.float64))


def run_ours(args):
    import numpy as np
    import torch
    from alphazero_risk_b200 import api

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dist, azd = None, None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # the product's own multi-GPU entry points (az_dist_*, NCCL): rank 0's communicator id travels over the launcher's channel
        idt = torch.zeros(api.DIST_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(api.Dist.unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, src=0)
        azd = api.Dist(world_size=world, rank=rank, unique_id=bytes(idt.cpu().numpy().tobytes()), device=local)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    n, S = args.games, args.lockstep
    stream = torch.cuda.current_stream()
    sptr = stream.cuda_stream
    env = api.Env(n, device=local, first_game_id=rank * n)       # weak scaling: every rank owns n games, global ids rank*n ..
    env.reset(SEED, stream=sptr)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # > 126 MB L2

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        # the timed region below lasts tens of milliseconds, nvidia-smi samples every 100 ms: run the same launches (untimed) until the
        # sampler has seen the GPU under this load, so the clocks line describes the state the timed launches run in
        t_lead = time.perf_counter()
        while len(sampler.lines) < 3 and time.perf_counter() - t_lead < 3.0:
            env.rollout(S, stream=sptr)
            torch.cuda.synchronize()
    # the lead-in ran a time-dependent number of moves: deal again, so that every run with the same arguments times the same games
    env.reset(SEED, stream=sptr)
    for _ in range(args.warmup):
        env.rollout(S, stream=sptr)
    torch.cuda.synchronize()
    env.counters(reset=True, stream=sptr)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(i & 0xff)                 # L2 flush between timed iterations (untimed)
        ev[i][0].record(stream)
        env.rollout(S, stream=sptr)
        ev[i][1].record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    cnt = env.counters(stream=sptr)
    assert cnt["steps"] == n * S * args.steps, cnt
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env, cnt, sptr)

    # ---- e2e: host State images in pinned memory -> device -> rollout -> host, every step.  The public calls are synchronous
    # (az_env_import_aos / az_env_rollout / az_env_export_aos return when the data is there), so a host that wants the copies of one
    # shard to overlap the rollout of another drives shards from separate threads, each with its own env handle and stream: here
    # --e2e-shards shards (default 4; swept 2 / 3 / 4 / 8 on B200: 12.1 / 12.3 / 12.4 / 8.3 G steps/s) of games/shards.  Every step of a shard continues from the images its previous step exported.
    e2e_steps = max(3, min(args.steps, 10))
    n_sh = max(1, args.e2e_shards)
    per = n // n_sh
    shards = []
    for k in range(n_sh):
        st = torch.cuda.Stream()
        e = api.Env(per, device=local, first_game_id=rank * n + k * per)
        h_a = torch.empty((per, 160), dtype=torch.uint8).pin_memory()
        h_b = torch.empty((per, 160), dtype=torch.uint8).pin_memory()
        e.reset(SEED, stream=st.cuda_stream)
        e.export_aos(out=h_a.numpy(), stream=st.cuda_stream)
        shards.append([e, st, h_a, h_b])

    def e2e_shard(sh, steps):
        e, st, h_in, h_out = sh
        torch.cuda.set_device(local)
        for _ in range(steps):
            e.import_aos(h_in.numpy(), stream=st.cuda_stream)
            e.rollout(S, stream=st.cuda_stream)
            e.export_aos(out=h_out.numpy(), stream=st.cuda_stream)
            e.counters(stream=st.cuda_stream)
            h_in, h_out = h_out, h_in
        sh[2], sh[3] = h_in, h_out

    def e2e_run(steps):
        th = [threading.Thread(target=e2e_shard, args=(sh, steps)) for sh in shards]
        for t in th:
            t.start()
        for t in th:
            t.join()

    e2e_run(2)
    barrier()
    t0 = time.perf_counter()
    e2e_run(e2e_steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_games = per * n_sh
    for sh in shards:
        sh[0].close()

    dev_ms, e2e_ms, wall_ms = dev_ms, e2e_s * 1e3, t_wall * 1e3
    if dist is not None:
        from alphazero_risk_b200 import dist as azdist
        dev_ms, e2e_ms, wall_ms = azdist.max_over_ranks([dev_ms, e2e_ms, wall_ms], dist)
        cnt = azd.gather_counters([cnt])                  # az_dist_gather_counters (GameResults::add over the ranks)

    mcts_line = None
    if not args.no_selfplay:
        mcts_line = run_selfplay(args, api, torch, dist, azd, rank, world, local, barrier)
    # BASELINE configs[4]'s per-GPU shape (16384 games x 800 simulations, one move after one warm-up move) and the CMake-default
    # 20-block graph at configs[2]'s shape: sub-lines of the same JSON line, at every N
    cfg5_line = blocks20_line = None
    if not args.no_selfplay and args.cfg5_games > 0:
        cfg5_line = run_selfplay(args, api, torch, dist, azd, rank, world, local, barrier, label="configs[4] per-GPU shape", with_tree=False,
                                 shape=(args.cfg5_games, args.cfg5_sims, args.blocks, 1, 1, 1))
    if not args.no_selfplay and args.blocks20:
        blocks20_line = run_selfplay(args, api, torch, dist, azd, rank, world, local, barrier, label="configs[2] shape, CMake-default graph",
                                     with_tree=False, shape=(args.sp_games, args.sp_sims, 20, 1, 2, 1))

    play_line = None
    if args.play_games >= 2 and rank == 0 and world == 1:
        play_line = run_play(args, api, torch, rank, local)

    train_line = None
    if args.train_batch >= 2 and rank == 0 and world == 1:
        train_line = run_train(args, api, torch, local)
    env6_line = None
    if args.env6_games > 0 and rank == 0:
        env6_line = run_env6(args, api, torch, rank, local)
    cfg4_line = None
    if not args.no_selfplay and args.cfg4_games > 0:
        cfg4_line = run_selfplay6(args, api, torch, dist, azd, rank, world, local, barrier)

    if rank == 0:
        hbm_peak, _, src = measured_peaks()
        env_traffic = ncu_traffic("k_env_rollout")
        if env_traffic["traffic"] is not None:
            env_traffic["dram_achieved"] = env_traffic["traffic"] / (dev_ms / args.steps * 1e-3) / 1e9        # GB/s really moved
        cap, why = ncu_capture("k_env_rollout")
        if cap is not None and "issue_active_pct" in cap:
            # the roofline that can still move: thread-instructions issued per cycle against 4 schedulers x 32 lanes per SM
            ia, lanes = cap["issue_active_pct"] / 100.0, cap["lanes_per_inst"]
            env_issue = {"bound": "issue", "issue_slots_busy": ia, "active_lanes_per_instruction": lanes, "lanes": 32,
                         "frac": ia * lanes / 32.0, "warps_active_pct": cap.get("warps_active_pct"), "capture": cap.get("capture"),
                         "note": "ncu --set full of this binary's k_env_rollout (sources hash-checked): fraction of the SM's lane-issue "
                                 "capacity doing game work = issue slots busy x active lanes / 32; 65536 games are only 13.8 warps per SM"}
        else:
            env_issue = {"bound": "issue", "frac": None, "stale": why}
        total_steps = n * S * args.steps * world
        value = total_steps / (dev_ms * 1e-3)
        kernel_ms = dev_ms / args.steps
        achieved = ENV_BYTES_PER_STEP * n * S / (kernel_ms * 1e-3) / 1e9
        line = dict(metric="env_steps_per_sec", value=value, unit="steps/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=kernel_ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="u8", data="synthetic",
                    config=dict(env_config(n, S), l2="256 MiB flush between timed iterations",
                                sharding="games by contiguous global id, no data-path collective"),
                    roofline=dict({"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                                   "algorithmic_bytes_per_launch": ENV_BYTES_PER_STEP * n * S, "peak_source": src,
                                   "note": "achieved = ALGORITHMIC bytes (330 B/step x games x moves per launch, SURVEY 8d) / CUDA-event time of "
                                           "k_env_rollout, as the metric contract asks; it is NOT the kernel's DRAM rate: the state stays on chip "
                                           "for the moves of a launch (traffic = ncu DRAM bytes of one launch, dram_achieved = traffic / time), "
                                           "so the kernel is bound by instruction issue / latency — see issue_roofline; for the same reason frac is not capped at 1"},
                                  **env_traffic),
                    issue_roofline=env_issue,
                    e2e={"value": e2e_games * S * e2e_steps * world / (e2e_ms * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": e2e_games * 160,
                         "d2h_bytes_per_step": e2e_games * 160 + 64 * n_sh, "steps": e2e_steps,
                         "note": "%d host threads x %d games, each: import State images (pinned host) -> 512-move rollout -> export images + "
                                 "counters, every step; one shard's copies overlap the others' rollouts" % (n_sh, per)},
                    gpu_launches=args.steps, wall_ms_timed_region=wall_ms, clocks=clocks,
                    results={"games_finished": cnt["games"], "wins": cnt["wins"], "draws": cnt["draws"]})
        if mcts_line is not None:
            line["mcts"] = mcts_line
            line["gpu_launches"] += mcts_line["gpu_launches"]
        for key, sub in (("cfg5", cfg5_line), ("blocks20", blocks20_line), ("cfg4", cfg4_line)):
            if sub is not None:
                line[key] = sub
                line["gpu_launches"] += sub["gpu_launches"]
        if play_line is not None:
            line["play"] = play_line
        if train_line is not None:
            line["train"] = train_line
        if env6_line is not None:
            line["env6"] = env6_line
            line["gpu_launches"] += env6_line["gpu_launches"]
        if world == 1 and not args.no_cpu_baseline:
            cb, _ = cpu_env_baseline(12.0)
            line["cpu_baseline"] = cb
            if mcts_line is not None:
                mcts_line["cpu_baseline"] = cpu_selfplay_baseline(args.sp_sims, 10.0)
        print(json.dumps(line))
    env.close()
    if azd is not None:
        azd.close()
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed rollout launches of the headline line; its e2e sub-line times max(3, min(K, 10)) steps and the self-play "
                         "sub-line max(2, min(K, --sp-steps))")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--games", type=int, default=65536)
    ap.add_argument("--lockstep", type=int, default=512, help="lockstep moves per launch (one bench step)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-shards", type=int, default=4, help="host threads (each with its own env shard and stream) of the e2e measurement")
    ap.add_argument("--no-selfplay", action="store_true", help="skip the configs[2] self-play measurement")
    ap.add_argument("--sp-games", type=int, default=4096)
    ap.add_argument("--sp-sims", type=int, default=64)
    ap.add_argument("--sp-moves", type=int, default=2, help="self-play moves per timed step")
    ap.add_argument("--sp-steps", type=int, default=4, help="max timed self-play steps")
    ap.add_argument("--sp-descents", type=int, default=1, help="az_rules.concurrent_descents for the self-play measurement")
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--cfg5-games", type=int, default=16384, help="games per GPU of the configs[4] sub-line (0 skips it)")
    ap.add_argument("--cfg5-sims", type=int, default=800)
    ap.add_argument("--cfg4-games", type=int, default=16384, help="games per GPU of the six-player self-play sub-line (configs[3]; 0 skips it)")
    ap.add_argument("--cfg4-sims", type=int, default=200)
    ap.add_argument("--env6-games", type=int, default=16384, help="games of the six-player environment sub-line (configs[3]'s game; 0 skips it)")
    ap.add_argument("--no-blocks20", dest="blocks20", action="store_false", help="skip the 20-block (CMake default graph) sub-line")
    ap.add_argument("--train-batch", type=int, default=512, help="training-step measurement batch (SETTINGS.BATCH_SIZE); 0 skips it")
    ap.add_argument("--play-games", type=int, default=1000, help="configs[0] match size (--cg); 0 skips it")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write rank 0's game State images and the counters "
                                                          "of the timed steps to DIR/*.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    # stdout carries the ONE JSON line and nothing else: whatever libraries write to file descriptor 1 meanwhile (NCCL prints its
    # version banner there) goes to stderr
    sys.stdout.flush()
    _json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = _json_out
    main()
    _json_out.flush()
