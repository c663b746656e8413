#!/usr/bin/env python
"""bench.py -- self-play moves/sec (8x8, 800 sims) on N B200s, plus env steps/sec (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[2] -- 8x8 board, default 128x10 network with the
reference's random initialisation (torch.manual_seed(0)), 800 MCTS simulations per move, 4,096 concurrent
self-play games per GPU.  One timed "step" = one move for every game slot = 4,096 full searches
(801 leaf evaluations each) + action selection + state update, all enqueued by ONE C-ABI call
(yy_selfplay_run).  value = moves/s of the whole job, state resident in HBM.  e2e = the same metric through
the host-buffer search API (numpy boards in -> H2D -> 800-sim search -> visit counts D2H -> host-side action
choice -> host-buffer state update), copies inside the timed region.  Weak scaling: 4,096 games per GPU at
every N (N=8 is configs[3]'s 32,768 games); games are independent, so there is no data-path collective --
NCCL only broadcasts the packed weight image before, and gathers replay records after, the timed region.

--impl reference times the reference's CPU implementation of the same path (oracle/port.py, kind "port":
the upstream code is pure Python and cannot travel to the GPU box) with one worker process per host core.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS = COLS = 8
GAMES_PER_GPU = 4096
SIMS = 800
CHANNELS, BLOCKS = 128, 10
A = ROWS * COLS
# algorithmic FLOPs (2*MAC) per leaf evaluation, SURVEY 8d / BASELINE.md section 3
FLOPS_TOWER_PER_BOARD = 2 * A * (9 * 5 * CHANNELS + BLOCKS * 2 * 9 * CHANNELS * CHANNELS + CHANNELS * 64)   # conv layers
FLOPS_PER_LEAF = FLOPS_TOWER_PER_BOARD + 2 * (32 * A * A + 32 * A * 256 + 256)                               # + FC heads = 380,584,448
ENV_BYTES_PER_STEP = 6 * ((A + 7) // 8) + 4                                                                  # 52 B
ENV_BOARDS = 65536


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile(prefix="yyclk", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = sorted(s for s, p in zip(sm, pw) if p > 0.5 * max(pw)) or sorted(sm)
        return {"sm_mhz": busy[len(busy) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw)}


# ------------------------------------------------------------------------------------------------ reference arm / cpu baseline
PLY_SPREAD = 40        # CPU samples search positions after 0..39 random plies: with rolling games the GPU arm's timed region (25 launches of
                       # one search budget each at the driver's arguments) takes a slot through ~37 moves


def cpu_selfplay_sample(workers, searches_per_worker=1, sims=SIMS, rows=ROWS, cols=COLS):
    """(moves/s, cores, description): oracle port, one process per core, 1 torch thread each.  Worker i searches (as
    player 1, like self_play.py:135) the position reached after (i * 25) // workers uniformly random legal plies."""
    from oracle import port
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    jobs = [(rows, cols, sims, searches_per_worker, CHANNELS, BLOCKS, 1, i, (i * PLY_SPREAD) // workers) for i in range(workers)]
    with ctx.Pool(workers) as pool:
        times = pool.map(port._worker, jobs)
    total = workers * searches_per_worker
    return total / max(times), workers, (f"{total} searches of {sims} sims on {rows}x{cols} from random-play positions at plies 0..{PLY_SPREAD - 1} "
                                        f"(one per worker), {workers} worker processes x 1 torch thread (reference scaling axis: --workers), "
                                        f"slowest worker {max(times):.1f}s, fastest {min(times):.1f}s")


def cpu_env_sample(workers, steps_per_worker=1500):
    """(steps/s one core, steps/s all cores): the reference's Python env loop (getValidMoves + getNextState + getGameEnded,
    random play; oracle/port.py env_steps) on one core and on one process per core."""
    from oracle import port
    import multiprocessing as mp
    t0 = time.perf_counter()
    port.env_steps(ROWS, COLS, steps_per_worker, seed=0)
    one = steps_per_worker / (time.perf_counter() - t0)
    ctx = mp.get_context("spawn")
    with ctx.Pool(workers) as pool:
        times = pool.map(port._env_worker, [(ROWS, COLS, steps_per_worker, i) for i in range(workers)])
    return one, workers * steps_per_worker / max(times)


def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_workers():
    return max(1, min(cpu_cores(), 64))


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    workers = cpu_workers()
    vals = []
    t_all = time.perf_counter()
    for i in range(args.warmup + args.steps):
        v, cores, sample = cpu_selfplay_sample(workers, 1, SIMS)
        if i >= args.warmup:
            vals.append(v)
    value = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": "self-play moves/sec (8x8, 800 sims)", "value": value, "unit": "moves/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * workers / value,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": "moves/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "moves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t_all}
    emit(line)


def workload_config(n_gpus):
    return {"workload": f"BASELINE.json configs[2]: 8x8, {SIMS} sims/move, {GAMES_PER_GPU} concurrent self-play games per GPU, "
                        f"128ch x 10 residual blocks, reference random init (torch.manual_seed(0)); weak scaling",
            "board": "8x8", "sims_per_move": SIMS, "games_per_gpu": GAMES_PER_GPU, "global_games": GAMES_PER_GPU * n_gpus,
            "network": "128x10", "parallelism": f"games sharded over {n_gpus} GPU(s), no data-path collective",
            "step": f"one launch of the persistent kernel = {SIMS + 1} evaluation steps (the budget of one full search) for every game slot; "
                    "games are rolling (a slot whose search is complete makes its move and starts the next search at once), so the moves a "
                    "step completes are counted by the device, not assumed",
            "semantics": "deterministic sequential MCTS per game (1 leaf/game/step), search-as-black (reference self_play.py:99,135)",
            "l2_policy": "inputs larger than L2: per step the kernels stream 801 x 7.3 MB of weights from L2 and the tree arenas (3.8 GB) live in HBM"}


def flops_per_leaf(rows, cols):
    A_ = rows * cols
    return 2 * A_ * (9 * 5 * CHANNELS + BLOCKS * 2 * 9 * CHANNELS * CHANNELS + CHANNELS * 64) + 2 * (32 * A_ * A_ + 32 * A_ * 256 + 256)


# ------------------------------------------------------------------------------------------------ B200 arm
def timed_rolling(eng, torch, dist, world, iters, warmup, steps, barrier):
    """warmup + steps launches of `iters` evaluation steps; returns (ms max over ranks, moves of all ranks, evaluations of
    this rank, kernel profile of this rank), all inside the timed region."""
    for _ in range(warmup):
        eng.selfplay_advance(iters)
    barrier()
    st0 = eng.stats()
    eng.set_profiling(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        eng.selfplay_advance(iters)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    prof = eng.get_profile()
    eng.set_profiling(False)
    st = eng.stats()
    moves, evals = st.moves - st0.moves, st.tower_evals - st0.tower_evals
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        t = torch.tensor([moves], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        moves = int(t.item())
    return ms, moves, evals, prof, st


def tensor_roofline(peaks, evals, prof, ms, flops_leaf, extra=None):
    tower_s = prof["ms"] * 1e-3 / max(1, prof["launches"])
    per_launch = evals / max(1, prof["launches"])
    achieved = flops_leaf * per_launch / tower_s / 1e12 if prof["launches"] else None
    roof = {"bound": "tensor", "kernel": "fused_kernel (persistent search: tower + FC heads + tree step + episode driver, yy_fused.cu)",
            "achieved": achieved, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
            "frac": (achieved / peaks["bf16_tflops_sustained"]) if achieved else None,
            "peak_source": f"bf16_tflops_sustained of {peaks['source']} (kernel timed inside a long step)",
            "launches_timed": prof["launches"], "avg_launch_ms": tower_s * 1e3, "share_of_step": prof["ms"] / ms if ms else None,
            "algorithmic_flops_per_launch": flops_leaf * per_launch, "leaf_evaluations_per_launch": per_launch,
            "evaluations": "required ones only: the kernel evaluates a board only when a game has a pending leaf (device counter "
                           "tower_evals = leaves requested by the searches + their roots)"}
    if extra:
        roof.update(extra)
    return roof


DUMP_BYTES = 64 << 20


def dump_outputs(engine, eng, plies, out_dir):
    """Writes the replay records (Engine.replay_window: board before the move, root visit counts, game serial, ply, player)
    that the timed self-play holds after its last step, with the result code of each record's game from the results
    table, as float32 / float64 .npy files under out_dir, sorted by (game serial, ply).

    The records kept are those of the games the reset starts (serials 0 .. n_games - 1) at plies 0 .. plies - 1, so that
    runs with the same arguments write the same records.  That set does not depend on timing: a search needs at most
    SIMS + 1 evaluation steps and a finished search moves in the same step, so after L launches of SIMS + 1 steps every
    slot has made at least L moves (the caller passes L - 1); the content of a record depends only on the seed, the game
    serial and the ply.  Which records a given launch appends does depend on timing: simulations that end in revisited
    terminals are advanced by background warps while the tower runs.  For the same reason a game that goes on past the
    kept plies may or may not be over when the run stops, so its result code is written as 0 (not over by the last kept
    ply); only games that end within the kept plies carry their code.  Above DUMP_BYTES a fixed, seeded sample is written."""
    import numpy as np
    from yinyang_game_alphazero_b200 import bitboard
    n = eng.stats().examples
    if n > eng.replay_capacity:
        raise RuntimeError(f"replay ring wrapped ({n} records, capacity {eng.replay_capacity}): the first games are gone")
    rec = eng.replay_window(0, n)
    results = engine._to_host(eng.replay_views()["results"])[0]
    serial, ply = rec["game_serial"].astype(np.int64), rec["ply"].astype(np.int64)
    keep = np.flatnonzero((serial >= 0) & (serial < eng.n_games) & (ply < plies))
    keep = keep[np.lexsort((ply[keep], serial[keep]))]
    code = results[serial % len(results)]
    per_game = np.bincount(serial[keep], minlength=eng.n_games)
    short = np.flatnonzero(per_game != plies)
    if len(np.unique(serial[keep] * plies + ply[keep])) != len(keep) or np.any(code[keep][np.isin(serial[keep], short)] == 0) \
            or np.any(per_game[short] == 0):
        raise RuntimeError(f"the first {eng.n_games} games do not all hold plies 0..{plies - 1} (or their whole game)")
    first = (serial >= 0) & (serial < eng.n_games)
    ended_within = np.bincount(serial[first], minlength=eng.n_games) <= plies     # every move of the game is a kept record
    code = np.where(first & ended_within[np.where(first, serial, 0)], code, 0)
    out = {"boards": bitboard.unpack_boards(rec["black"], rec["white"], ROWS, COLS).astype(np.float32),
           "visit_counts": rec["counts"].astype(np.float32),
           "game_serial": serial.astype(np.float64),
           "ply": ply.astype(np.float32),
           "player": rec["player"].astype(np.float32),
           "game_result": code.astype(np.float32)}
    per_record = sum(a[0].nbytes for a in out.values())
    if len(keep) * per_record > DUMP_BYTES:
        keep = keep[np.sort(np.random.default_rng(0).choice(len(keep), DUMP_BYTES // per_record, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a[keep])


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import yy_b200  # noqa: F401
    from yinyang_game_alphazero_b200 import engine, weights, distributed as yyd
    from yinyang_game_alphazero_b200 import network

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # weights: reference init on rank 0, packed, broadcast over NCCL (north star: weights broadcast)
    torch.manual_seed(0)
    sd = network._Params(ROWS, COLS, CHANNELS, BLOCKS).state_dict()   # reference layout + initialisation (neural_network.py:39-92)
    iters = SIMS + 1
    eng = engine.Engine(rows=ROWS, cols=COLS, n_games=GAMES_PER_GPU, n_sims=SIMS, evaluator="nn", state_dict=sd,
                        seed=0xC0FFEE + rank, replay_capacity=GAMES_PER_GPU * (2 * (args.steps + args.warmup) + 8))
    t_bcast = t_bcast_first = 0.0
    if world > 1:
        t_bcast_first = yyd.broadcast_weights(eng)     # first collective of the process: NCCL sets its communicator up here
        t_bcast = yyd.broadcast_weights(eng)           # the 7.3 MB broadcast itself

    launches1 = engine._lib.lib().yy_launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    ms, moves, evals_timed, prof, st = timed_rolling(eng, torch, dist, world, iters, args.warmup, args.steps, barrier)
    clocks = sampler.stop()
    launches = engine._lib.lib().yy_launch_count() - launches1 - 2 * args.warmup
    value = moves / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(engine, eng, max(1, args.warmup + args.steps - 1), args.dump_outputs)

    # replay gather (north star: gather replay samples over NCCL), outside the timed region
    t_gather, n_records = (yyd.gather_replay_counts(eng) if world > 1 else (0.0, min(st.examples, eng.replay_capacity)))

    # ---- e2e: the same rolling self-play with HOST buffers: per step the packed weight image goes host -> device (pinned) and every
    # example the step produced comes back device -> host (positions, visit counts, game ids, results), all inside the timed region.
    # The read-back of step k runs on a second stream while step k + 1 computes (a stream-ordered snapshot of the device counters
    # taken right after step k says which records are complete).
    # A fresh engine with the same seed replays the same games, and the timed region covers the same steps as `value` (the rate
    # depends on the ply: searches late in a game revisit terminal nodes and need fewer evaluations).
    boards, players = eng.live_boards()
    players_s = np.ones_like(players)
    eng.search_host(boards, players_s)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(2):
        eng.search_host(boards, players_s)              # the host-buffer SEARCH API (MCTS.search for a batch): numpy boards in, visit counts out
    search_api = 2 * GAMES_PER_GPU / (time.perf_counter() - t0)
    eng.close(); del eng
    torch.cuda.empty_cache()
    eng = engine.Engine(rows=ROWS, cols=COLS, n_games=GAMES_PER_GPU, n_sims=SIMS, evaluator="nn", state_dict=sd,
                        seed=0xC0FFEE + rank, replay_capacity=GAMES_PER_GPU * (2 * (args.steps + args.warmup) + 8))
    e2e_steps = args.steps
    img_host = weights.pack_state_dict(sd, ROWS, COLS)
    pinned = torch.from_numpy(img_host).pin_memory()
    rec_bytes = 2 * 8 * eng.W + 2 * A + 4 + 2 + 1
    side = torch.cuda.Stream()
    snaps = [torch.empty(7, dtype=torch.int64, pin_memory=True) for _ in range(2)]
    evs = [torch.cuda.Event() for _ in range(2)]
    sview = eng.stats_view()
    state = {"cursor": eng.stats().examples, "d2h": 0, "records": 0}

    def launch(k):
        eng.weight_image.copy_(pinned, non_blocking=True)           # H2D: this step's input (the network the games are played with)
        eng.selfplay_advance(iters)
        snaps[k & 1].copy_(sview, non_blocking=True)                # which records exist once step k is complete
        evs[k & 1].record()

    def drain(k):
        evs[k & 1].synchronize()
        stop = int(snaps[k & 1][3])
        with torch.cuda.stream(side):
            rec = eng.replay_window(state["cursor"], stop)          # D2H: the step's examples (pinned staging, side stream)
            res = engine._to_host(eng.replay_views()["results"])[0]
        state["d2h"] += (stop - state["cursor"]) * rec_bytes + res.nbytes
        state["records"] += len(rec["ply"])
        state["cursor"] = stop

    for k in range(args.warmup):                                    # untimed, like the device leg: the first W moves of the games
        launch(k); drain(k)
    barrier()
    state.update(d2h=0, records=0)
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        launch(k)
        if k > 0:
            drain(k - 1)
    drain(e2e_steps - 1)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_moves, d2h = state["records"], state["d2h"]
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
        t = torch.tensor([e2e_moves], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        e2e_moves = int(t.item())
    e2e_value = e2e_moves / e2e_s
    eng.close(); del eng
    torch.cuda.empty_cache()

    # ---- the other BASELINE.json configurations (rank 0; 2 steps each), a strong-scaled configs[3] line, a tree-only leg
    other = {}
    if not args.quick:
        # configs[4] on ALL ranks (16x16, 1,600 sims, 4,096 games per GPU: at 8 GPUs the 32,768 games of the config)
        c4 = bench_config(engine, network, torch, peaks, 16, 1600, 4096, steps=2, iters=801, dist=dist if world > 1 else None, world=world,
                          barrier=barrier, seed=7 + rank)
        if rank == 0:
            other[f"configs[4] 16x16/1600 sims, 4,096 games per GPU x {world} GPU(s)"] = c4
            other["configs[0] 6x6/100 sims"] = bench_config(engine, network, torch, peaks, 6, 100, 4096, steps=3, iters=8 * 101)
            other["tree only (stub evaluator) 8x8/800"] = bench_tree_only(engine, torch, peaks)
    strong = None
    if world > 1 and not args.quick:
        strong = bench_strong(engine, torch, dist, world, rank, sd, peaks, barrier)

    # ---- env steps/s (BASELINE.json configs[1]): 65,536 synthetic random-play boards on this GPU
    full = rank == 0 and not args.quick
    env = bench_env(engine, torch, peaks) if full else None
    dataset = bench_dataset(engine, torch, peaks) if full else None
    learner_leg = bench_learner(engine, torch, peaks) if full else None
    learner_dp = bench_learner_dp(engine, torch, world) if world > 1 and not args.quick else None     # every rank takes part (NCCL all-reduce)
    if learner_leg is not None and learner_dp is not None:
        learner_leg["data_parallel"] = learner_dp
    ai_move_leg = bench_ai_move() if full else None

    if rank == 0:
        traffic = None
        tp = os.path.join(ROOT, "profiles", "tower_traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        roof = tensor_roofline(peaks, evals_timed, prof, ms, FLOPS_PER_LEAF, {"traffic": traffic})
        cpu = None
        if world == 1 and not args.no_cpu_baseline and not args.quick:
            v, cores, sample = cpu_selfplay_sample(cpu_workers(), 1, SIMS)
            cpu = {"value": v, "unit": "moves/s", "cores": cores, "kind": "port", "sample": sample}
            one, allc = cpu_env_sample(cpu_workers())
            env["cpu_baseline"] = {"value": allc, "unit": "steps/s", "cores": cpu_workers(), "kind": "port", "one_core": one,
                                   "sample": "1,500 random-play env steps (mask + step + ended) per worker process, oracle/port.py env_steps"}
        line = {"metric": "self-play moves/sec (8x8, 800 sims)", "value": value, "unit": "moves/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": workload_config(world), "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "moves/s", "h2d_bytes_per_step": int(img_host.nbytes), "d2h_bytes_per_step": int(d2h // e2e_steps),
                        "steps": e2e_steps, "moves": int(e2e_moves), "seconds": e2e_s,
                        "api": "Engine.selfplay_advance with host buffers: weight image H2D from pinned memory, every example of "
                               "the step D2H (Engine.replay_window + results table) while the next step computes; same games and "
                               "the same steps as `value` (fresh engine, same seed, same warm-up)",
                        "search_api": {"value": search_api, "unit": "moves/s", "api": "Engine.search_host (numpy boards in, visit counts out; lock-step batch of 4,096 searches)"}},
                "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "env": env, "dataset": dataset, "learner": learner_leg, "ai_move": ai_move_leg,
                "moves_per_s_roofline": peaks["bf16_tflops_sustained"] * 1e12 / ((SIMS + 1) * FLOPS_PER_LEAF) * world,
                "moves_per_s_roofline_note": "at SIMS + 1 evaluations per move; a search whose simulations revisit terminal nodes needs fewer (evals_per_move)",
                "leaf_evals_per_s": evals_timed * world / (ms * 1e-3), "moves_timed": int(moves), "evals_per_move": evals_timed * world / max(1, moves),
                "other_configs": other, "strong_scaling_configs3": strong,
                "nccl": {"weight_broadcast_s": t_bcast, "first_collective_s": t_bcast_first, "replay_gather_s": t_gather, "replay_records_gathered": int(n_records)},
                "selfplay_stats": st.__dict__}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def bench_config(engine, network, torch, peaks, n, sims, games, steps, iters, dist=None, world=1, barrier=None, seed=7):
    """Rolling self-play on another BASELINE.json geometry: moves/s (all ranks) and the roofline of required evaluations (this rank)."""
    torch.manual_seed(0)
    sd = network._Params(n, n, CHANNELS, BLOCKS).state_dict()
    eng = engine.Engine(rows=n, cols=n, n_games=games, n_sims=sims, evaluator="nn", state_dict=sd, seed=seed,
                        replay_capacity=games * 64)
    ms, moves, evals, prof, st = timed_rolling(eng, torch, dist, world, iters, 1, steps, barrier or torch.cuda.synchronize)
    fl = flops_per_leaf(n, n)
    out = {"board": f"{n}x{n}", "sims_per_move": sims, "games": games * world, "n_gpus": world, "value": moves / (ms * 1e-3), "unit": "moves/s", "steps": steps,
           "evaluation_steps_per_launch": iters, "ms_per_step": ms / steps, "evals_per_move": evals * world / max(1, moves),
           "roofline": tensor_roofline(peaks, evals, prof, ms, fl), "moves_per_s_roofline_at_sims_plus_1": world * peaks["bf16_tflops_sustained"] * 1e12 / ((sims + 1) * fl),
           "arena_gb": eng.workspace_bytes / 1e9, "overflow": st.overflow}
    eng.close(); del eng
    torch.cuda.empty_cache()
    return out


def bench_tree_only(engine, torch, peaks):
    """The tree kernels alone (north star: HBM GB/s for the tree kernels): the same persistent kernel with the deterministic-prior
    evaluator, i.e. expand + backup + select of 4,096 games per step and nothing else."""
    eng = engine.Engine(rows=ROWS, cols=COLS, n_games=GAMES_PER_GPU, n_sims=SIMS, evaluator="stub", seed=3, replay_capacity=GAMES_PER_GPU * 64)
    for _ in range(2):
        eng.selfplay_advance(SIMS + 1)
    torch.cuda.synchronize()
    s0 = eng.stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(4):
        eng.selfplay_advance(SIMS + 1)
    ev1.record(); torch.cuda.synchronize()
    s1 = eng.stats()
    sec = ev0.elapsed_time(ev1) * 1e-3
    sims, evals = s1.sims - s0.sims, s1.tower_evals - s0.tower_evals
    # algorithmic bytes per simulation (DESIGN 3.2): per level 20 B per child read (N, W, P, summary), 21 B per child written at the
    # expanded leaf, 8 B per path edge updated, node + leaf records; measured average below from the device's own counters is not
    # available, so the figure uses the survey's mid-game estimate of 3 KB per simulation
    bytes_per_sim = 3000.0
    gbs = sims * bytes_per_sim / sec / 1e9
    eng.close(); del eng
    torch.cuda.empty_cache()
    tt = None
    tp = os.path.join(ROOT, "profiles", "tree_traffic.json")
    if os.path.exists(tp):
        tt = json.load(open(tp))
    return {"value": sims / sec, "unit": "simulations/s", "leaves_per_s": evals / sec, "moves_per_s": (s1.moves - s0.moves) / sec,
            "roofline": {"bound": "hbm", "kernel": "fused_kernel with the stub evaluator (tree_step_game only)", "achieved": gbs, "peak": peaks["hbm_gbs"],
                         "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"], "traffic": tt,
                         "note": "~3 KB of algorithmic traffic per simulation (SURVEY 8d), served by L2: ncu measures 265 B of DRAM traffic per "
                                 "simulation (traffic: profiles/tree_traffic.json); pointer chasing, one dependent round trip per tree level, latency "
                                 "bound -- inside the real search these steps overlap the tower of the other games"}}


def bench_strong(engine, torch, dist, world, rank, sd, peaks, barrier):
    """BASELINE.json configs[3] as written: 32,768 concurrent games in total, sharded over the N GPUs (16,384 / 8,192 / 4,096 each)."""
    games = 32768 // world
    eng = engine.Engine(rows=ROWS, cols=COLS, n_games=games, n_sims=SIMS, evaluator="nn", state_dict=sd, seed=0xBEEF + rank,
                        replay_capacity=games * 16)
    ms, moves, evals, prof, st = timed_rolling(eng, torch, dist, world, SIMS + 1, 1, 2, barrier)
    out = {"total_games": 32768, "games_per_gpu": games, "n_gpus": world, "value": moves / (ms * 1e-3), "unit": "moves/s", "steps": 2,
           "ms_per_step": ms / 2, "scaling": "strong", "arena_gb_per_gpu": eng.workspace_bytes / 1e9,
           "roofline_rank0": tensor_roofline(peaks, evals, prof, ms, FLOPS_PER_LEAF), "overflow": st.overflow}
    eng.close(); del eng
    torch.cuda.empty_cache()
    return out


def bench_env(engine, torch, peaks):
    import numpy as np
    plies = torch.arange(ENV_BOARDS, dtype=torch.int32) % 52
    black0, white0, players0 = engine.random_playout(ENV_BOARDS, plies, ROWS, COLS, seed=0xC0FFEE)
    mask0 = engine.legal_mask(black0, white0, players0, ROWS, COLS)
    from yinyang_game_alphazero_b200 import bitboard
    bits = bitboard.unpack_bits(mask0.cpu().numpy().view(np.uint64), ROWS, COLS)
    acts_h = np.where(bits.any(axis=1), bits.argmax(axis=1), -1).astype(np.int32)   # lowest legal move, else -1
    acts = torch.from_numpy(acts_h).cuda()
    out_mask, out_res = torch.empty_like(black0), torch.empty_like(players0)
    reps, inner = 20, 8
    bufs = [(black0.clone(), white0.clone(), players0.clone()) for _ in range(inner)]
    for b, w, p in bufs[:3]:
        engine.env_step(b, w, p, acts, ROWS, COLS, out_mask=out_mask, out_result=out_res)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total_ms = 0.0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for r in range(reps):
        bufs = [(black0.clone(), white0.clone(), players0.clone()) for _ in range(inner)]
        flush.fill_(r)                                  # L2 flush: write a buffer larger than L2 (126 MB)
        torch.cuda.synchronize()
        ev0.record()
        for b, w, p in bufs:
            engine.env_step(b, w, p, acts, ROWS, COLS, out_mask=out_mask, out_result=out_res)
        ev1.record(); torch.cuda.synchronize()
        total_ms += ev0.elapsed_time(ev1)
    api_launch_s = total_ms * 1e-3 / (reps * inner)      # one Python/ctypes call per launch: bound by the host's issue rate
    # the same 8 launches replayed from a CUDA graph (fresh boards restored and L2 flushed before every replay): device time
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for b, w, p in bufs:
            engine.env_step(b, w, p, acts, ROWS, COLS, out_mask=out_mask, out_result=out_res)
    total_ms = 0.0
    for r in range(reps):
        for b, w, p in bufs:
            b.copy_(black0); w.copy_(white0); p.copy_(players0)
        flush.fill_(r)
        torch.cuda.synchronize()
        ev0.record()
        graph.replay()
        ev1.record(); torch.cuda.synchronize()
        total_ms += ev0.elapsed_time(ev1)
    per_launch_s = total_ms * 1e-3 / (reps * inner)
    steps_s = ENV_BOARDS / per_launch_s
    # e2e: host buffers
    boards = bitboard.unpack_boards(black0.cpu().numpy().view(np.uint64), white0.cpu().numpy().view(np.uint64), ROWS, COLS)
    pl, ac = players0.cpu().numpy(), acts.cpu().numpy()
    engine.env_step_host(boards, pl, ac, ROWS, COLS)
    t0 = time.perf_counter()
    for _ in range(3):
        engine.env_step_host(boards, pl, ac, ROWS, COLS)
    e2e = 3 * ENV_BOARDS / (time.perf_counter() - t0)
    hbk, hwh = black0.cpu().numpy().view(np.uint64), white0.cpu().numpy().view(np.uint64)
    engine.env_step_host_packed(hbk, hwh, pl, ac, ROWS, COLS)
    t0 = time.perf_counter()
    for _ in range(5):
        engine.env_step_host_packed(hbk, hwh, pl, ac, ROWS, COLS)
    e2e_packed = 5 * ENV_BOARDS / (time.perf_counter() - t0)
    gbs = ENV_BYTES_PER_STEP * ENV_BOARDS / per_launch_s / 1e9
    # the same kernel on a batch large enough to fill the machine (16 x the config): throughput rather than latency
    big = 16 * ENV_BOARDS
    pb = torch.arange(big, dtype=torch.int32) % 52
    bb, wb, plb = engine.random_playout(big, pb, ROWS, COLS, seed=0xC0FFEE)
    ab = acts.repeat(16)
    omb, orb = torch.empty_like(bb), torch.empty_like(plb)
    copies = [(bb.clone(), wb.clone(), plb.clone()) for _ in range(4)]
    engine.env_step(*copies[0], ab, ROWS, COLS, out_mask=omb, out_result=orb)
    torch.cuda.synchronize()
    ev0.record()
    for b, w, p in copies[1:]:
        engine.env_step(b, w, p, ab, ROWS, COLS, out_mask=omb, out_result=orb)
    ev1.record(); torch.cuda.synchronize()
    big_s = ev0.elapsed_time(ev1) * 1e-3 / 3
    return {"metric": "env steps/sec (8x8)", "workload": "BASELINE.json configs[1]: 65,536 synthetic random-play boards, fused mask+step+ended",
            "value": steps_s, "unit": "steps/s", "us_per_launch": per_launch_s * 1e6,
            "timing": "8 launches replayed from a CUDA graph, CUDA events around the replay",
            "per_call": {"value": ENV_BOARDS / api_launch_s, "unit": "steps/s", "us_per_launch": api_launch_s * 1e6,
                         "note": "one engine.env_step() Python/ctypes call per launch, device-resident tensors"},
            "e2e": {"value": e2e_packed, "unit": "steps/s", "api": "env_step_host_packed (packed uint64 boards in host memory in and out: 21 B in, 34 B out per board)",
                    "h2d_bytes_per_step": 21, "d2h_bytes_per_step": 34,
                    "int8_arrays": {"value": e2e, "unit": "steps/s", "api": "env_step_host (the reference's int8[n,m] board arrays in/out; bit packing on the device)"}},
            "roofline": {"bound": "hbm", "kernel": "env_step_kernel", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": gbs / peaks["hbm_gbs"], "traffic": 1.384e6,
                         "note": "3.4 MB of algorithmic traffic per launch; a launch of ONE block costs 2.0-2.2 us (launch + cold-DRAM "
                                 "latency, tools/env_floor.py), the rest is integer issue (two lanes per board, line-fill connectivity, "
                                 "437 warp instructions per 16 boards); integer-issue bound when the machine is full; traffic = DRAM "
                                 "bytes of one launch (the boards are read once, the outputs are still in L2 when it ends; "
                                 "profiles/r02_env_step_sq_ncu_summary.txt)"},
            "saturated": {"boards": big, "value": big / big_s, "unit": "steps/s", "us_per_launch": big_s * 1e6,
                          "achieved_GBps": ENV_BYTES_PER_STEP * big / big_s / 1e9},
            "l2_policy": "L2 flushed (256 MB write) before each timed group of 8 launches on fresh boards"}


_JSON_FD = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else any library prints (NCCL's version banner,
    torchrun notices) was redirected to stderr in main()."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def bench_dataset(engine, torch, peaks):
    """SURVEY 8f-1: replay records -> training tensors with the 8-fold augmentation (yy_augment_samples), HBM bound."""
    n_rec = 262144                                           # 3.2 GB of output per launch: far larger than L2
    plies = torch.arange(n_rec, dtype=torch.int32) % 52
    black, white, _ = engine.random_playout(n_rec, plies, ROWS, COLS, seed=0xDA7A)
    counts = torch.randint(0, 800, (n_rec, A), dtype=torch.int16, device="cuda")
    values = torch.ones(n_rec, dtype=torch.float32, device="cuda")
    out = engine.augment_samples(black, white, ROWS, COLS, counts=counts, values=values)
    torch.cuda.synchronize()
    # caller-allocated outputs, as over the C ABI (yy_augment_samples writes into the caller's buffers); one event pair per launch
    reps = 9
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    evs[0].record()
    for k in range(reps):
        engine.augment_samples(black, white, ROWS, COLS, counts=counts, values=values, out=out)
        evs[k + 1].record()
    torch.cuda.synchronize()
    per = sorted(evs[k].elapsed_time(evs[k + 1]) for k in range(reps))
    sec = per[reps // 2] * 1e-3
    del out
    # the same call with torch allocating the 3.2 GB of outputs each time (what a caller without buffers of its own pays)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(5):
        o = engine.augment_samples(black, white, ROWS, COLS, counts=counts, values=values)
        del o
    ev1.record(); torch.cuda.synchronize()
    sec_alloc = ev0.elapsed_time(ev1) * 1e-3 / 5
    bytes_per_record = 16 + 2 * A + 4 + 8 * (6 * A + 1) * 4
    gbs = bytes_per_record * n_rec / sec / 1e9
    return {"metric": "augmented training samples/sec (8x8, 8 forms per replay record)", "value": 8 * n_rec / sec, "unit": "samples/s",
            "records": n_rec, "ms_per_launch": sec * 1e3, "ms_per_launch_all": per, "ms_per_call_with_output_allocation": sec_alloc * 1e3,
            "roofline": {"bound": "hbm", "kernel": "augment_kernel", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": gbs / peaks["hbm_gbs"], "traffic": 3.209e9, "algorithmic_bytes_per_record": bytes_per_record,
                         "note": "write-only stream; the peak is the measured read+write copy rate, which a pure write stream can exceed; "
                                 "traffic = dram read + write of one launch (profiles/r01_augment_v2_ncu_summary.txt)"},
            "l2_policy": "outputs (3.2 GB per launch) larger than L2; median of 9 launches into caller-allocated outputs"}


def bench_learner_dp(engine, torch, world):
    """Data-parallel learner over all ranks (weak scaling: batch 64 per GPU): every step = backward graph, one NCCL
    all-reduce of the 14.5 MB flat gradient buffer, Adam graph.  Max over ranks of the device time."""
    import torch.distributed as dist
    from yinyang_game_alphazero_b200 import learner as lrn, network
    B = 64
    torch.manual_seed(0)
    net = network._Params(ROWS, COLS, 128, 10)
    rank = dist.get_rank()
    plies = torch.arange(B, dtype=torch.int32) % 52
    black, white, _ = engine.random_playout(B, plies, ROWS, COLS, seed=0x1EA2 + rank)
    counts = torch.randint(0, 800, (B, A), dtype=torch.int16, device="cuda")
    values = torch.ones(B, device="cuda")
    planes, pol, val = engine.augment_samples(black, white, ROWS, COLS, counts=counts, values=values)
    L = lrn.Learner(ROWS, COLS, 128, 10, batch_size=B, state_dict=net.state_dict(), data_parallel=True)
    for _ in range(4):
        L.step(planes[:B], pol[:B], val[:B])
    torch.cuda.synchronize(); dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 32
    ev0.record()
    for i in range(steps):
        j = (i % 8) * B
        L.step(planes[j:j + B], pol[j:j + B], val[j:j + B])
    ev1.record(); torch.cuda.synchronize()
    t = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = float(t.item()) * 1e-3 / steps
    w0 = L.params[:1024].clone()
    dist.broadcast(w0, 0)
    return {"value": world * B / sec, "unit": "samples/s", "ms_per_step": sec * 1e3, "n_gpus": world, "scaling": "weak",
            "weights_identical_across_ranks": bool(torch.equal(w0, L.params[:1024])),
            "collective": "one NCCL all-reduce of the flat gradient buffer (%.1f MB) per step" % (L.grads.numel() * 4 / 1e6)}


def bench_ai_move():
    """SURVEY 8f-4: latency of one AI move as the GUI requests it (src/gui/server.py:30-129: one position, 100 simulations,
    reference-initialised 128x10 network), through ai_move.get_ai_move with host dictionaries in and out."""
    import tempfile
    import numpy as np
    from yinyang_game_alphazero_b200 import ai_move
    from yinyang_game_alphazero_b200.game import YinYangGame
    from yinyang_game_alphazero_b200.network import YinYangNeuralNetwork
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "best_model.pth.tar")
        YinYangNeuralNetwork(YinYangGame(ROWS, COLS)).save_model(path)
        board = np.zeros((ROWS, COLS), np.int8); board[3, 3] = 1; board[3, 4] = -1
        req = {"board": board.tolist(), "currentPlayer": 1, "rows": ROWS, "cols": COLS, "modelPath": path}
        ai_move.get_ai_move(req)                               # builds the engine, loads the weights
        times = []
        for _ in range(10):
            t0 = time.perf_counter()
            out = ai_move.get_ai_move(req)
            times.append(time.perf_counter() - t0)
        ai_move.get_ai_move(req, num_threads=8)                # mcts_threads = 8: 8 leaves per step with virtual loss
        times8 = []
        for _ in range(10):
            t0 = time.perf_counter()
            out8 = ai_move.get_ai_move(req, num_threads=8)
            times8.append(time.perf_counter() - t0)
    return {"metric": "AI move latency (8x8, 100 simulations, one position)", "value": float(np.median(times) * 1e3), "unit": "ms",
            "higher_is_better": False, "valid_move": bool(out.get("validMove")), "api": "ai_move.get_ai_move (request / response dictionaries of /api/ai_move)",
            "mcts_threads_8": {"value": float(np.median(times8) * 1e3), "unit": "ms", "valid_move": bool(out8.get("validMove")),
                               "note": "num_threads=8 -> 8 simulations per network batch (virtual loss), the counterpart of mcts.py:414-426"}}


def bench_learner(engine, torch, peaks):
    """SURVEY 8f-2: optimisation steps of the reference trainer (trainer.py:120-137; batch 64, Adam) on the 128x10 network,
    8x8 boards: one CUDA-graph replay of the yy_lrn_* kernels per step.  Tensor bound on paper, latency bound in fact."""
    import numpy as np
    from yinyang_game_alphazero_b200 import learner as lrn, _lib, network
    B = 64
    torch.manual_seed(0)
    net = network._Params(ROWS, COLS, 128, 10)                 # reference layout + initialisation
    n_rec = 256
    plies = torch.arange(n_rec, dtype=torch.int32) % 52
    black, white, _ = engine.random_playout(n_rec, plies, ROWS, COLS, seed=0x1EA2)
    counts = torch.randint(0, 800, (n_rec, A), dtype=torch.int16, device="cuda")
    values = (torch.randint(0, 2, (n_rec,), device="cuda").float() * 2 - 1)
    planes, pol, val = engine.augment_samples(black, white, ROWS, COLS, counts=counts, values=values)   # 2,048 samples
    out = {}
    for precision in ("3xtf32", "tf32"):
        L = lrn.Learner(ROWS, COLS, 128, 10, batch_size=B, state_dict=net.state_dict(), precision=precision, data_parallel=False)
        l0 = _lib.lib().yy_launch_count()
        first = L.step(planes[:B], pol[:B], val[:B]).clone()
        kernels = (_lib.lib().yy_launch_count() - l0) // 2     # the eager step + its capture pass both count
        for i in range(1, 4):
            L.step(planes[i * B:(i + 1) * B], pol[i * B:(i + 1) * B], val[i * B:(i + 1) * B])
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = 64
        ev0.record()
        for i in range(steps):
            j = (i % 32) * B
            last = L.step(planes[j:j + B], pol[j:j + B], val[j:j + B])
        ev1.record(); torch.cuda.synchronize()
        sec = ev0.elapsed_time(ev1) * 1e-3 / steps
        flops = 3 * B * FLOPS_PER_LEAF                           # forward + backward-data + backward-weights (algorithmic)
        tf = flops / sec / 1e12
        peak = peaks["bf16_tflops_sustained"] / 2                # TF32 runs at half the bf16 rate; no measured TF32 peak on file
        out[precision] = {"value": B / sec, "unit": "samples/s", "ms_per_step": sec * 1e3, "kernels_per_step": int(kernels),
                          "losses_first": [float(x) for x in first.tolist()], "losses_last": [float(x) for x in last.tolist()],
                          "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak, "traffic": None,
                                       "peak_source": "half of the measured sustained bf16 rate (TF32 = half rate)",
                                       "algorithmic_flops_per_step": flops,
                                       "note": "4,096 positions per step: every kernel is microseconds long, the step is launch/latency bound"}}
    # the same step at batch 512 (8 x the positions per kernel): how far the kernels are from their roofline once they are
    # not microseconds long (the reference's batch size stays the headline)
    Bl = 512
    for precision in ("3xtf32", "tf32"):
        Ll = lrn.Learner(ROWS, COLS, 128, 10, batch_size=Bl, state_dict=net.state_dict(), precision=precision, data_parallel=False)
        for i in range(3):
            Ll.step(planes[i * Bl:(i + 1) * Bl], pol[i * Bl:(i + 1) * Bl], val[i * Bl:(i + 1) * Bl])
        torch.cuda.synchronize()
        ev0.record()
        for i in range(16):
            j = (i % 4) * Bl
            Ll.step(planes[j:j + Bl], pol[j:j + Bl], val[j:j + Bl])
        ev1.record(); torch.cuda.synchronize()
        sec_l = ev0.elapsed_time(ev1) * 1e-3 / 16
        tf_l = 3 * Bl * FLOPS_PER_LEAF / sec_l / 1e12
        out[precision]["batch_512"] = {"value": Bl / sec_l, "unit": "samples/s", "ms_per_step": sec_l * 1e3, "achieved_tflops": tf_l,
                                       "frac_of_tf32_roofline": tf_l / (peaks["bf16_tflops_sustained"] / 2),
                                       "library_baseline": "stock PyTorch 2.11 eager on the same B200 (tools/torch_learner_baseline.py): 17.8 ms fp32, 7.2 ms with TF32 convolutions"}
        del Ll
    # end to end through the reference-facing trainer: host examples in (boards, policies, values), device dataset
    # construction + augmentation, shuffled batches, checkpoint-ready weights out
    from yinyang_game_alphazero_b200 import trainer as trn
    from yinyang_game_alphazero_b200.game import YinYangGame
    import tempfile
    game = YinYangGame(ROWS, COLS)
    rng = np.random.default_rng(0)
    grids = (rng.integers(0, 3, (512, ROWS, COLS)) - 1).astype(np.int8)
    pis = rng.random((512, A)); pis /= pis.sum(1, keepdims=True)
    examples = [(grids[i], pis[i], float(rng.choice([-1.0, 1.0]))) for i in range(512)]
    with tempfile.TemporaryDirectory() as d:
        tr = trn.AlphaZeroTrainer(game, model_dir=d, batch_size=B, data_parallel=False)
        tr.train(examples[:64], epochs=1, augment=True)        # graph capture
        t0 = time.perf_counter()
        m = tr.train(examples, epochs=2, augment=True)         # 4,096 samples x 2 epochs = 128 steps
        e2e_s = time.perf_counter() - t0
    out["3xtf32"]["e2e"] = {"value": 2 * 8 * len(examples) / e2e_s, "unit": "samples/s", "steps": 128,
                            "h2d_bytes_per_step": B * (2 * 8 + 4 * A + 4) // 8, "d2h_bytes_per_step": 0,
                            "api": "AlphaZeroTrainer.train(examples, epochs=2, augment=True): host examples in, metrics out",
                            "total_loss_per_epoch": [float(x) for x in m["total_loss"]]}
    # CPU baseline: the same step as the reference runs it (oracle/port.py training_step = trainer.py:120-137 in fp32 torch),
    # on this box's host cores with torch's own intra-op threading
    from oracle import port                                    # cpu_baseline leg: the one place the bench runs the oracle
    cpu_net = port.build_net(ROWS, COLS, 128, 10)
    cpu_opt = torch.optim.Adam(cpu_net.parameters(), lr=1e-3, weight_decay=1e-4)
    hp, hq, hv = planes[:B].cpu(), pol[:B].cpu(), val[:B].cpu()
    port.training_step(cpu_net, cpu_opt, hp, hq, hv)
    t0 = time.perf_counter()
    for _ in range(3):
        port.training_step(cpu_net, cpu_opt, hp, hq, hv)
    cpu_s = (time.perf_counter() - t0) / 3
    out["3xtf32"]["cpu_baseline"] = {"value": B / cpu_s, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
                                     "sample": "3 optimisation steps of batch 64 (fp32 torch on the host, intra-op threads = cores)"}
    res = out["3xtf32"]
    res["metric"] = "training samples/sec (8x8, 128x10 network, batch 64, Adam; one CUDA-graph replay per step)"
    res["single_pass_tf32"] = out["tf32"]
    res["l2_policy"] = "a step touches ~190 MB of activations, im2col scratch, weights and Adam state (> L2); 32 distinct batches rotate"
    return res


def main():
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="developer runs: only the self-play legs (value, e2e, roofline)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the replay records of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
