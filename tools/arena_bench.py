#!/usr/bin/env python
"""Wall time of the current-vs-best arena (arena.py, DESIGN.md §3.5): one command, one JSON file.

    python tools/arena_bench.py [--out profiles/arena_bench.json]

Workload: 8x8, two 128x10 networks with the reference's initialisation (torch.manual_seed(0) and (1)), 400 simulations.
  (a) arena.play_match, 16 games from the empty board: two batched searches per ply, host round trip between plies;
  (b) arena.DeviceArena, the same 16 games (openings 0) on the persistent kernel, both models in one launch per ply --
      its results and plies must equal (a) game for game;
  (c) arena.DeviceArena, 256 games from paired 8-ply random openings (make_openings), with the count of distinct starts
      (opening x colour assignment).
Each leg is timed with a host clock around the call, which ends in a device synchronise; engine construction is not
timed (nor the packing of the weight images).  A short warm-up of both paths runs first.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, power, clk = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def main(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "arena_bench.json"))
    p.add_argument("--sims", type=int, default=400)
    args = p.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("arena_bench needs a CUDA device")
    import yy_b200  # noqa: F401
    from yinyang_game_alphazero_b200 import arena, engine, network, weights
    from yinyang_game_alphazero_b200.game import YinYangGame
    from yinyang_game_alphazero_b200.mcts import MCTS
    game = YinYangGame(8, 8)
    sds = []
    for seed in (0, 1):
        torch.manual_seed(seed)
        sds.append(network._Params(8, 8, 128, 10).state_dict())
    imgs = [engine.device_image(weights.pack_state_dict(sd, 8, 8), torch.cuda.current_device()) for sd in sds]
    res = {"card": card(), "workload": f"8x8, 128x10 (reference init, seeds 0 and 1), {args.sims} simulations"}

    def host(G, sims):
        mc = []
        for sd in sds:
            net = network.YinYangNeuralNetwork(game, 128, 10)
            net.load_state_dict(sd)
            mc.append(MCTS(game, net, num_simulations=sims, verbose=0))
            mc[-1]._engine(G)                                                   # engine construction is not timed
        try:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = arena.play_match(game, mc[0], mc[1], G)
            torch.cuda.synchronize()
            return out, time.perf_counter() - t0
        finally:
            for m in mc:
                m.close()

    def device(G, sims, openings=None):
        a = arena.DeviceArena(game, G, sims, 128, 10)
        try:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = a.play(imgs[0], imgs[1], openings)
            torch.cuda.synchronize()
            return out, time.perf_counter() - t0
        finally:
            a.close()

    host(2, 8)
    device(2, 8)
    ha, ta = host(16, args.sims)
    print("a", ta, ha["plies"].tolist(), flush=True)
    hb, tb = device(16, args.sims)
    print("b", tb, hb["plies"].tolist(), flush=True)
    same = bool(np.array_equal(ha["results"], hb["results"]) and np.array_equal(ha["plies"], hb["plies"])
                and all(ha[k] == hb[k] for k in ("current_wins", "best_wins", "draws")))
    op = arena.make_openings(game, 256, 8, seed=0)
    hc, tc = device(256, args.sims, op)
    print("c", tc, flush=True)
    starts = {(bytes(op["black"][i]), bytes(op["white"][i]), int(op["player"][i]), bool(op["a_plays_black"][i])) for i in range(256)}

    def leg(out, s, G):
        return {"games": G, "seconds": s, "plies_total": int(out["plies"].sum()), "plies_max": int(out["plies"].max()),
                "current_wins": out["current_wins"], "best_wins": out["best_wins"], "draws": out["draws"],
                "win_ratio": out["win_ratio"]}
    res["a_play_match_16"] = leg(ha, ta, 16)
    res["b_device_arena_16"] = {**leg(hb, tb, 16), "equals_a": same}
    res["c_device_arena_256_openings8"] = {**leg(hc, tc, 256), "distinct_starts": len(starts)}
    res["speedup_b_over_a"] = ta / tb
    res["ratio_c_over_b"] = tc / tb
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "speedup_b_over_a", "ratio_c_over_b")}))
    print(json.dumps(res["b_device_arena_16"]))
    if not same:
        raise SystemExit("the device arena's games differ from play_match's")


if __name__ == "__main__":
    main()
