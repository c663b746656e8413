"""Playout cap randomisation of self-play on the GPU (yy_selfplay_set_playout_cap, DESIGN.md §3.3): off is bit-identical,
whole capped games equal the oracle's game with the same fast / full plies, games do not depend on the slot or the
driver, plain searches ignore the cap, bad arguments are refused, and the Python drivers count games without records."""
import math

import numpy as np
import pytest

import playout_cap_ref as P
from conftest import randomise_bn

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng(yy):
    from yinyang_game_alphazero_b200 import engine
    return engine


def _nn_state(n, m, seed=11):
    import torch
    from oracle import port
    torch.manual_seed(seed)
    return randomise_bn(port.build_net(n, m, 128, 1)).state_dict()


def _run_quota(e, total, chunk):
    """Rolling self-play until `total` games (the quota) are finished; then every slot idles."""
    e.selfplay_set_quota(total)
    for _ in range(4000):
        e.selfplay_advance(chunk)
        if e.stats().games_finished >= total:
            break
    st = e.stats()
    assert st.games_finished == total and st.overflow == 0 and st.examples <= e.replay_capacity
    return st


def _records(e):
    """{serial: [(ply, board bytes, counts bytes, player)] sorted by ply}"""
    rp = e.replay()
    games = {}
    for i in np.lexsort((rp["ply"], rp["game_serial"])):
        games.setdefault(int(rp["game_serial"][i]), []).append(
            (int(rp["ply"][i]), rp["boards"][i].tobytes(), rp["counts"][i].tobytes(), int(rp["player"][i])))
    return games, rp


def _results(e, total):
    """result code of every game serial < total (the results table)"""
    res = e.replay_views()["results"].cpu().numpy()
    return res[np.arange(total) % len(res)].tolist()


def _stat_tuple(st):
    return (st.moves, st.evals, st.games_finished, st.examples, st.sims, st.overflow, st.max_depth, st.tower_evals)


# ------------------------------------------------------------------------------------------------ 1. off = bit-identical
@pytest.mark.parametrize("evaluator", ["stub", "nn"])
def test_cap_off_is_bit_identical(eng, evaluator):
    """selfplay_set_playout_cap(1.0, k) leaves the records, the results table and the stats exactly as without the call."""
    n = m = 6
    total, sims = 24, 30
    kw = {"state_dict": _nn_state(n, m)} if evaluator == "nn" else {}
    runs = []
    for call in (False, True):
        e = eng.Engine(rows=n, cols=m, n_games=8, n_sims=sims, evaluator=evaluator, seed=31, replay_capacity=total * 200, **kw)
        if call:
            e.selfplay_set_playout_cap(1.0, 5)
        st = _run_quota(e, total, 211)
        games, _ = _records(e)
        runs.append((games, _results(e, total), _stat_tuple(st)))
        e.close()
    assert runs[0] == runs[1]
    assert runs[0][2][0] == runs[0][2][3]                  # moves == examples


def _by_game_ply(ex):
    """play()'s examples in (game, ply) order: each drain is sorted, but which drain a game's records arrive in depends on
    how far the launches got"""
    order = np.lexsort((ex["ply"], ex["game"]))
    return {k: v[order] for k, v in ex.items()}


def test_cap_off_rolling_selfplay_is_bit_identical(yy):
    """RollingSelfPlay with full_search_prob=1.0 returns the same examples (and leaves the same stats) as without it."""
    from yinyang_game_alphazero_b200.game import YinYangGame
    from yinyang_game_alphazero_b200.self_play import RollingSelfPlay
    out = []
    for kw in ({}, {"full_search_prob": 1.0, "fast_simulations": 3}):
        sp = RollingSelfPlay(YinYangGame(5, 5), slots=8, num_simulations=20, seed=9, evaluator="stub", **kw)
        ex = _by_game_ply(sp.play(20))
        out.append((ex, _stat_tuple(sp.eng.stats())))
        sp.close()
    (a, sa), (b, sb) = out
    assert sa == sb and sorted(a) == sorted(b)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


# ------------------------------------------------------------------------------------------------ 2. whole games vs the oracle
def _capped_games_vs_oracle(eng, n, m, sims, tt, sab, p_full, fast, total=48, slots=16, seed=0):
    A, PL = n * m, 4 * n * m
    rng = np.random.default_rng(n * 100 + m)
    uniforms = rng.random((total, PL))
    noise = np.stack([rng.dirichlet([0.3] * A) for _ in range(total)])
    e = eng.Engine(rows=n, cols=m, n_games=slots, n_sims=sims, evaluator="stub", temperature_threshold=tt, search_as_black=sab,
                   replay_capacity=total * PL, seed=seed)
    e.selfplay_set_random_stream(uniforms, noise)
    e.selfplay_set_playout_cap(p_full, fast)
    st = _run_quota(e, total, 701)
    rp = e.replay()
    results = _results(e, total)
    e.close()
    order = np.lexsort((rp["ply"], rp["game_serial"]))
    n_full = n_fast = 0
    ply0 = set()
    empty_games = 0
    for s in range(total):
        b, pi, z, kind, full_plies, fast_plies, result = P.play_game(
            n, m, sims, uniforms[s], noise[s], temperature_threshold=tt, search_as_black=sab,
            playout_cap=(fast, lambda step, s=s: P.full(seed, s, step, p_full)))
        idx = order[rp["game_serial"][order] == s]
        assert rp["ply"][idx].tolist() == full_plies, s                 # the recorded plies are the full ones
        assert np.array_equal(rp["boards"][idx], b), s
        assert np.array_equal(rp["pi"][idx], pi), s                      # float64, bit for bit
        assert np.array_equal(rp["z"][idx], z), s
        assert eng.result_from_code(results[s]) == result, s           # defined for games without records too
        n_full += len(full_plies); n_fast += len(fast_plies)
        ply0.add(0 in full_plies)
        empty_games += not full_plies
    assert (st.examples, st.moves - st.examples) == (n_full, n_fast)
    assert st.tower_evals == st.evals + st.moves
    return ply0, empty_games, n_fast


@pytest.mark.parametrize("fast", ["quarter", "one"])
@pytest.mark.parametrize("n,m,sims,tt,sab", [(4, 4, 50, 3, True), (6, 6, 40, 8, True), (5, 7, 30, 10, True), (8, 8, 24, 10, True),
                                             (6, 6, 40, 8, False)])
def test_capped_episodes_match_oracle(eng, n, m, sims, tt, sab, fast):
    """48 whole games on 16 slots at p_full = 0.5, recorded stream: per game the recorded plies, boards, pi and z equal the
    oracle's game with the same full / fast plies; moves - examples is the number of fast plies.  Both a full and a fast
    ply 0 occur (the noise and the no-noise root)."""
    fast_sims = sims // 4 if fast == "quarter" else 1
    ply0, _, n_fast = _capped_games_vs_oracle(eng, n, m, sims, tt, sab, 0.5, fast_sims)
    assert ply0 == {True, False} and n_fast > 0


def test_capped_games_without_records_match_oracle(eng):
    """p_full = 0.05 on 4x4: some finished games have no record at all; their results (and every other game) still match."""
    _, empty_games, _ = _capped_games_vs_oracle(eng, 4, 4, 50, 3, True, 0.05, 12)
    assert empty_games >= 1


# ------------------------------------------------------------------------------------------------ 3. slot independence
def test_capped_games_do_not_depend_on_the_slot(eng):
    """nn evaluator, cap on: 40 games on 8 slots with launch boundaries mid-search equal 40 games on 40 slots."""
    n = m = 6
    total, sims = 40, 30
    sd = _nn_state(n, m)
    runs = []
    for slots, chunk in ((8, 97), (40, 1000)):
        e = eng.Engine(rows=n, cols=m, n_games=slots, n_sims=sims, evaluator="nn", seed=77, replay_capacity=total * 400, state_dict=sd)
        e.selfplay_set_playout_cap(0.5, 8)
        st = _run_quota(e, total, chunk)
        e.selfplay_advance(50)                           # quota used up: every slot idles
        assert _stat_tuple(e.stats()) == _stat_tuple(st)
        assert st.tower_evals == st.evals + st.moves and 0 < st.examples < st.moves
        games, _ = _records(e)
        runs.append((games, _results(e, total), st.moves, st.examples))
        e.close()
    assert runs[0] == runs[1]
    assert all(r != 0 for r in runs[0][1])


# ------------------------------------------------------------------------------------------------ 4. lock-step = rolling
def test_capped_lockstep_matches_rolling(eng):
    """The per-step-kernel driver roots each search with the budget sp_prepare chose: every (game, ply) both drivers
    recorded is the same record."""
    n = m = 6
    slots, sims, moves = 24, 40, 45
    runs = []
    for sk in (False, True):
        e = eng.Engine(rows=n, cols=m, n_games=slots, n_sims=sims, evaluator="stub", seed=5, step_kernels=sk)
        e.selfplay_set_playout_cap(0.5, 6)
        e.selfplay_run(moves)
        st = e.stats()
        assert st.moves == slots * moves and st.overflow == 0 and 0 < st.examples < st.moves
        runs.append(_records(e)[0])
        e.close()
    ga, gb = runs
    common = 0
    for s in set(ga) & set(gb):
        k = min(len(ga[s]), len(gb[s]))
        assert ga[s][:k] == gb[s][:k], s
        common += k
    assert common >= slots * moves // 4


# ------------------------------------------------------------------------------------------------ 5. plain searches
@pytest.mark.parametrize("step_kernels", [False, True])
def test_plain_search_ignores_the_cap(eng, oracle_mod, step_kernels):
    """After fast self-play searches, Engine.search still runs n_sims simulations: the oracle's visit counts."""
    from conftest import random_play_boards
    n = m = 6
    games, sims = 12, 40
    boards, players = random_play_boards(oracle_mod, n, m, games, seed=4)
    e = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="stub", step_kernels=step_kernels)
    e.selfplay_set_playout_cap(0.0, 4)
    e.selfplay_run(3)                                   # the slots' last searches were fast ones (budget 4)
    assert e.stats().examples == 0
    counts, _ = e.search_host(boards, players)
    e.close()
    for g in range(games):
        r = oracle_mod.mcts_search(boards[g], int(players[g]), n, m, sims)
        assert np.array_equal(counts[g], r["counts"]), g


# ------------------------------------------------------------------------------------------------ 6. argument checks
def test_playout_cap_argument_checks(eng):
    e = eng.Engine(rows=4, cols=4, n_games=2, n_sims=10, evaluator="stub")
    for prob, fast in ((-0.1, 5), (1.5, 5), (math.nan, 5), (0.5, 0), (0.5, 11)):
        with pytest.raises(eng._lib.YinYangError):
            e.selfplay_set_playout_cap(prob, fast)
    e.selfplay_set_playout_cap(0.0, 10)
    e.selfplay_set_playout_cap(1.0, 1)
    e.close()
    x = eng.Engine(rows=4, cols=4, n_games=2, n_sims=10, evaluator="external")
    with pytest.raises(eng._lib.YinYangError):
        x.selfplay_set_playout_cap(0.5, 5)
    x.close()


# ------------------------------------------------------------------------------------------------ 7. Python drivers
def test_rolling_selfplay_play_counts_games_without_records(yy):
    """RollingSelfPlay.play(64) at p_full = 0.05: returns after exactly 64 finished games (many without a record) with
    exactly their full-search records: every record in the engine's ring, once each."""
    from yinyang_game_alphazero_b200.game import YinYangGame
    from yinyang_game_alphazero_b200.self_play import RollingSelfPlay
    sp = RollingSelfPlay(YinYangGame(4, 4), slots=16, num_simulations=24, seed=21, evaluator="stub", full_search_prob=0.05,
                         fast_simulations=4)
    ex = sp.play(64)
    st = sp.eng.stats()
    assert st.games_finished == 64 and sp.games_returned == 64
    assert len(ex["z"]) == st.examples and st.examples < st.moves
    assert len(np.unique(ex["game"])) < 64                      # some games have no record at all
    ex = _by_game_ply(ex)
    rp = sp.eng.replay()
    ring = np.lexsort((rp["ply"], rp["game_serial"]))
    assert np.array_equal(ex["game"], rp["game_serial"][ring]) and np.array_equal(ex["ply"], rp["ply"][ring])
    assert np.array_equal(ex["boards"], rp["boards"][ring]) and np.array_equal(ex["pi"], rp["pi"][ring])
    assert np.array_equal(ex["z"], rp["z"][ring]) and set(ex["game"].tolist()) <= set(range(64))
    key = ex["game"].astype(np.int64) * 4096 + ex["ply"]
    assert np.all(np.diff(key) > 0)                              # no record twice
    sp.close()


def test_device_loop_with_the_cap_records_full_searches_only(yy):
    import torch
    from yinyang_game_alphazero_b200.device_loop import DeviceLoop
    from yinyang_game_alphazero_b200.game import YinYangGame
    torch.manual_seed(0)
    loop = DeviceLoop(YinYangGame(4, 4), num_iterations=1, num_episodes=12, num_simulations=16, num_epochs=1, batch_size=32,
                      sample_size=256, eval_games=0, num_channels=32, num_res_blocks=1, slots=8, save_files=False, seed=1,
                      full_search_prob=0.3, fast_simulations=4)
    hist = loop.run()
    st = loop.selfplay.eng.stats()
    assert len(loop.buffer) == hist[0]["examples_global"] > 0
    assert hist[0]["examples_local"] <= st.examples < st.moves            # only recorded moves reach the buffer
    assert np.isfinite(hist[0]["policy_loss"])
    loop.close()
