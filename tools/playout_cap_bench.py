#!/usr/bin/env python
"""Throughput of playout cap randomisation (Engine.selfplay_set_playout_cap, DESIGN.md §3.3): one command, one JSON file.

    python tools/playout_cap_bench.py [--runs 3] [--out profiles/playout_cap_bench.json]

Workload: 8x8, 800 simulations, 4,096 rolling slots, the 128x10 network with the reference's initialisation
(torch.manual_seed(0)).  Two arms alternate: "off" (every move a full search) and "cap" (p_full 0.25, fast_sims 100).
- windowed: per fresh engine, 5 warm-up launches of selfplay_advance(801), then 20 timed ones (device events around the
  launches): searches/s, recorded examples/s, evaluations per search, evaluations per recorded example (evaluations =
  boards the persistent kernel evaluated, roots included);
- complete games: per arm, 4,096 whole games on 4,096 slots (RollingSelfPlay.play, what play_games_arrays runs; host
  clock around the call, which ends in a synchronise; engine construction not timed): finished games/s, examples per game.
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

ARMS = {"off": (1.0, None), "cap": (0.25, 100)}


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, power, clk = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def windowed(engine, torch, sd, arm, warm=5, steps=20, iters=801):
    p_full, fast = ARMS[arm]
    eng = engine.Engine(rows=8, cols=8, n_games=4096, n_sims=800, evaluator="nn", state_dict=sd, seed=0xC0FFEE,
                        replay_capacity=4096 * 16)
    if p_full != 1.0:
        eng.selfplay_set_playout_cap(p_full, fast)
    for _ in range(warm):
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
    searches, examples, evals = st.moves - st0.moves, st.examples - st0.examples, st.tower_evals - st0.tower_evals
    s = ms * 1e-3
    return {"ms": ms, "searches": searches, "examples": examples, "evaluations": evals, "games_finished": st.games_finished - st0.games_finished,
            "searches_per_s": searches / s, "examples_per_s": examples / s, "evals_per_search": evals / searches,
            "evals_per_example": evals / examples}


def complete_games(torch, sd, arm, games=4096):
    from yinyang_game_alphazero_b200.game import YinYangGame
    from yinyang_game_alphazero_b200.self_play import RollingSelfPlay
    p_full, fast = ARMS[arm]
    sp = RollingSelfPlay(YinYangGame(8, 8), sd, slots=games, num_simulations=800, seed=0xC0FFEE, full_search_prob=p_full,
                         fast_simulations=fast)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ex = sp.play(games)
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    st = sp.eng.stats()
    sp.close()
    assert st.games_finished == games
    return {"seconds": s, "games": games, "examples": int(len(ex["z"])), "searches": st.moves, "evaluations": st.tower_evals,
            "games_per_s": games / s, "examples_per_game": len(ex["z"]) / games, "searches_per_game": st.moves / games}


def main(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--runs", type=int, default=3)
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "playout_cap_bench.json"))
    args = p.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("playout_cap_bench needs a CUDA device")
    import yy_b200  # noqa: F401
    from yinyang_game_alphazero_b200 import engine, network
    res = {"card": card(), "workload": "8x8, 128x10 (reference init, torch.manual_seed(0)), 800 sims, 4096 rolling slots",
           "arms": {k: {"full_search_prob": v[0], "fast_simulations": v[1]} for k, v in ARMS.items()}}
    torch.manual_seed(0)
    sd = network._Params(8, 8, 128, 10).state_dict()
    win = {k: [] for k in ARMS}
    for _ in range(args.runs):
        for arm in ARMS:
            win[arm].append(windowed(engine, torch, sd, arm))
            print(arm, win[arm][-1], flush=True)
    keys = ("searches_per_s", "examples_per_s", "evals_per_search", "evals_per_example")
    res["windowed"] = {arm: {"runs": v, **{k: statistics.mean(r[k] for r in v) for k in keys}} for arm, v in win.items()}
    res["windowed_ratio_cap_over_off"] = {k: res["windowed"]["cap"][k] / res["windowed"]["off"][k] for k in keys}
    full = {}
    for arm in ARMS:
        full[arm] = complete_games(torch, sd, arm)
        print(arm, full[arm], flush=True)
    res["complete_games"] = full
    res["complete_games_ratio_cap_over_off"] = {k: full["cap"][k] / full["off"][k] for k in ("games_per_s", "examples_per_game")}
    res["strength"] = "not measured"
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "windowed_ratio_cap_over_off", "complete_games_ratio_cap_over_off")}))


if __name__ == "__main__":
    main()
