"""Host logic of the arena (no GPU): paired openings, the reference's accounting and the sharded arena's aggregation."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _arena():
    import yy_b200  # noqa: F401
    from yinyang_game_alphazero_b200 import arena, game
    return arena, game


def _fake_playout(count, plies, rows, cols, seed=0, rule_flags=0, device="cuda"):
    """Stand-in for engine.random_playout with its contract: board i depends only on (seed, i, plies[i])."""
    W = (rows * cols + 63) // 64
    i = np.arange(count, dtype=np.uint64)
    key = np.array([(seed * 0x9E3779B97F4A7C15 + k * 0xD1B54A32D192ED03 ^ int(plies[0])) % 2**64 for k in range(count)], np.uint64)
    black = np.stack([key >> np.uint64(w) for w in range(W)], axis=1)
    white = ~black
    return (torch.from_numpy(black.view(np.int64)), torch.from_numpy(white.view(np.int64)),
            torch.from_numpy(np.where(i % 2 == 0, 1, -1).astype(np.int8)))


def test_make_openings_pairs_colours_and_independence(monkeypatch):
    arena, game = _arena()
    g = game.YinYangGame(6, 6)
    monkeypatch.setattr(arena._engine, "random_playout", _fake_playout)
    a = arena.make_openings(g, 9, 4, seed=3)
    b = arena.make_openings(g, 20, 4, seed=3)
    for k in ("black", "white", "player", "a_plays_black"):
        assert np.array_equal(a[k], b[k][:9]), k                          # opening i does not depend on num_games
    assert np.array_equal(a["black"][0::2][:4], a["black"][1::2])         # games 2i and 2i+1 share opening i
    assert len({bytes(x) for x in a["black"][0::2]}) == 5                 # distinct pairs get distinct openings
    assert list(a["a_plays_black"]) == [i % 2 == 0 for i in range(9)]     # play_match's first_is_current
    c = arena.make_openings(g, 9, 4, seed=4)
    assert not np.array_equal(a["black"], c["black"])
    sh = arena.shard_openings(b, 4, 10)
    assert np.array_equal(sh["black"], b["black"][4:10]) and list(sh["a_plays_black"]) == [True, False] * 3


def test_make_openings_empty_boards():
    arena, game = _arena()
    g = game.YinYangGame(5, 7)
    o = arena.make_openings(g, 5, 0, seed=1)                              # no playout, no device
    assert o["black"].shape == (5, 1) and not o["black"].any() and not o["white"].any()
    assert np.all(o["player"] == 1) and list(o["a_plays_black"]) == [True, False, True, False, True]


def _reference_counts(results):
    """play_match's accounting before it moved into arena.tally (alphazero.py:206-222)."""
    G = len(results)
    first_is_current = (np.arange(G) % 2) == 0
    first_won, second_won = results == 1, results == -1
    cw = int(np.sum(first_won & first_is_current) + np.sum(second_won & ~first_is_current))
    bw = int(np.sum(first_won & ~first_is_current) + np.sum(second_won & first_is_current))
    return cw, bw, G - cw - bw


def test_tally_reproduces_play_match_accounting():
    arena, _ = _arena()
    rng = np.random.default_rng(0)
    for G in (0, 1, 2, 7, 40):
        for _ in range(20):
            res = rng.choice([1.0, -1.0, 0.0001, 0.0], size=G)
            t = arena.tally(res, (np.arange(G) % 2) == 0)
            assert (t["current_wins"], t["best_wins"], t["draws"]) == _reference_counts(res)
            assert t["win_ratio"] == (t["current_wins"] / G if G else 0.0)
    # the colours come from a_plays_black, not from the game index
    t = arena.tally(np.array([1.0, 1.0, -1.0]), np.array([False, True, False]))
    assert (t["current_wins"], t["best_wins"], t["draws"]) == (2, 1, 0)


def _synthetic(G):
    rng = np.random.default_rng(42)
    return rng.choice([1.0, -1.0, 0.0001], size=G)


def _stub_play(G):
    arena, _ = _arena()
    res = _synthetic(G)
    a_black = (np.arange(G) % 2) == 0
    return lambda lo, hi: arena.tally(res[lo:hi], a_black[lo:hi])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, G, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    arena, _ = _arena()
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        seen = []

        def play(lo, hi):
            seen.append((lo, hi))
            return _stub_play(G)(lo, hi)
        q.put((rank, arena.play_sharded(G, play, rank, world), seen))
    finally:
        dist.destroy_process_group()


def test_sharded_arena_world2_matches_one_rank():
    arena, _ = _arena()
    for G in (7, 8):
        one = arena.play_sharded(G, _stub_play(G))
        whole = arena.tally(_synthetic(G), (np.arange(G) % 2) == 0)
        assert one == whole
        world, port = 2, _free_port()
        ctx = mp.get_context("spawn")
        q = ctx.Queue()
        procs = [ctx.Process(target=_worker, args=(r, world, port, G, q)) for r in range(world)]
        for p in procs:
            p.start()
        res = sorted(q.get(timeout=120) for _ in range(world))
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
        (r0, out0, seen0), (r1, out1, seen1) = res
        assert out0 == out1 == one                                          # every rank gets the single-rank verdict
        (lo0, hi0), (lo1, hi1) = seen0[0], seen1[0]
        assert lo0 == 0 and hi0 == lo1 and hi1 == G and lo1 % 2 == 0       # whole pairs, contiguous, everything covered
