#!/usr/bin/env python
"""Cost of symmetric evaluation (Engine(eval_symmetry=)): one command, one JSON file.

    python tools/symmetry_bench.py [--runs 3] [--steps 3] [--out profiles/symmetry_bench.json]

- self-play throughput, 8x8 / 800 sims / 4,096 rolling games (bench.py's workload: 128x10 net with the reference's
  initialisation), eval_symmetry "none" and "random" alternating, `runs` fresh engines each; moves/s over `steps`
  launches of 801 evaluation steps after one warm-up launch (device events around the launches);
- AI-move latency: one game, 100 simulations, "none" against "average" at 8x8 and 6x6 (host clock around a search of
  device-resident roots that ends in a synchronise; median of 30 after 5 warm-up searches).
The card's name and power limit are read in the same run and written beside the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, power, clk = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def throughput(engine, torch, sd, sym, steps):
    iters = 801
    eng = engine.Engine(rows=8, cols=8, n_games=4096, n_sims=800, evaluator="nn", state_dict=sd, seed=0xC0FFEE,
                        replay_capacity=4096 * (2 * (steps + 1) + 8), eval_symmetry=sym)
    eng.selfplay_advance(iters)
    torch.cuda.synchronize()
    st0 = eng.stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        eng.selfplay_advance(iters)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    st = eng.stats()
    eng.close()
    moves, evals = st.moves - st0.moves, st.tower_evals - st0.tower_evals
    return {"moves_per_s": moves / (ms * 1e-3), "ms": ms, "moves": moves, "tower_evals": evals}


def latency(engine, torch, network, n, sym, reps=30, warm=5):
    from yinyang_game_alphazero_b200 import bitboard
    torch.manual_seed(0)
    sd = network._Params(n, n, 128, 10).state_dict()
    eng = engine.Engine(rows=n, cols=n, n_games=1, n_sims=100, evaluator="nn", state_dict=sd, replay_capacity=1,
                        eval_symmetry=sym, dirichlet_epsilon=0.0)
    board = torch.zeros((1, n, n), dtype=torch.int8)
    b, w = bitboard.pack_boards(board.numpy(), n, n)
    bd = torch.from_numpy(b.view("int64")).cuda()
    wd = torch.from_numpy(w.view("int64")).cuda()
    pd = torch.ones(1, dtype=torch.int8, device="cuda")
    out = torch.empty((1, n * n), dtype=torch.int32, device="cuda")
    ts = []
    for k in range(warm + reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.search(bd, wd, pd, out_counts=out)
        torch.cuda.synchronize()
        if k >= warm:
            ts.append((time.perf_counter() - t0) * 1e3)
    eng.close()
    return {"median_ms": statistics.median(ts), "min_ms": min(ts), "max_ms": max(ts), "reps": reps}


def main(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--runs", type=int, default=3)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "symmetry_bench.json"))
    args = p.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("symmetry_bench needs a CUDA device")
    import yy_b200  # noqa: F401
    from yinyang_game_alphazero_b200 import engine, network
    res = {"card": card(), "workload": "8x8, 128x10 (reference init, torch.manual_seed(0)), 800 sims, 4096 rolling games"}
    torch.manual_seed(0)
    sd = network._Params(8, 8, 128, 10).state_dict()
    tp = {"none": [], "random": []}
    for _ in range(args.runs):
        for sym in ("none", "random"):
            tp[sym].append(throughput(engine, torch, sd, sym, args.steps))
            print(sym, tp[sym][-1], flush=True)
    res["selfplay"] = {k: {"runs": v, "moves_per_s": [r["moves_per_s"] for r in v]} for k, v in tp.items()}
    res["selfplay_ratio_random_over_none"] = (statistics.mean(res["selfplay"]["random"]["moves_per_s"]) /
                                              statistics.mean(res["selfplay"]["none"]["moves_per_s"]))
    lat = {}
    for n in (8, 6):
        for rep in range(2):
            for sym in ("none", "average"):
                lat.setdefault(f"{n}x{n}", {}).setdefault(sym, []).append(latency(engine, torch, network, n, sym))
    res["ai_move_latency_100_sims"] = lat
    res["strength"] = "not measured"
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "selfplay_ratio_random_over_none")}))
    print(json.dumps(lat))


if __name__ == "__main__":
    main()
