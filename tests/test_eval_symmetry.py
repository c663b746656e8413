"""Symmetric evaluation on the GPU (Engine(eval_symmetry=), Engine.evaluate(form=)): a fixed form is the network on the
transformed board mapped back to the board's actions, averaging is the fp32 ascending-form mean of the fixed forms,
network-driven searches in random-form and averaged mode equal the oracle's search driven by the kernel's own
evaluate_form, and random-form rolling self-play is reproducible."""
import numpy as np
import pytest

import exact_net as X
import symmetry_ref as S
from conftest import random_play_boards, randomise_bn

pytestmark = pytest.mark.gpu

# one board per position layout (interleaved 8x8 / 6x6, half-board 16x16, row-aligned rectangular and square), an odd
# shape, a tall board whose group size is clamped, and a tiny one
BOARDS = [(8, 8, 128, 10), (6, 6, 128, 10), (16, 16, 128, 10), (10, 8, 128, 10), (12, 12, 128, 10), (5, 7, 64, 2),
          (32, 8, 128, 2), (3, 3, 32, 2)]
assert all(b in X.REPRESENTATIVES for b in BOARDS)


@pytest.fixture(scope="module")
def eng(yy):
    from yinyang_game_alphazero_b200 import engine
    return engine


@pytest.fixture(scope="module")
def sms(yy):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _net(n, m, channels, blocks, seed):
    import torch
    from oracle import port
    torch.manual_seed(seed)
    return randomise_bn(port.build_net(n, m, channels, blocks), seed=seed).state_dict()


def _batch(oracle_mod, n, m, count, seed):
    distinct, _ = random_play_boards(oracle_mod, n, m, 48, seed=seed, max_frac=0.7)
    rng = np.random.default_rng(seed)
    return distinct[rng.permutation(np.resize(np.arange(len(distinct)), count))]


@pytest.mark.parametrize("n,m,channels,blocks", BOARDS)
def test_fixed_form_is_the_transformed_board_mapped_back(eng, oracle_mod, host_tower_lib, sms, n, m, channels, blocks):
    """evaluate(b, form=f) == evaluate(T_f(b)) mapped back through form_src, bit for bit, for policy, value and logits;
    evaluate(b, form="average") == fp32 ascending-form mean of those.  Batches with partial groups and several heads
    batches per CTA; the averaged batch is larger than the engine's scratch holds, so it runs in chunks."""
    geo = X.tower_classes(host_tower_lib, n, m)
    sd = _net(n, m, channels, blocks, seed=n * 100 + m)
    big = sms * (geo["batch"] + 1) - 1
    e = eng.Engine(rows=n, cols=m, n_games=big, n_sims=1, evaluator="nn", state_dict=sd, replay_capacity=1)
    for count in (geo["Gb"] + 1, 2 * sms + 3, big):
        boards = _batch(oracle_mod, n, m, count, seed=count)
        per_form = []
        for f in S.forms(n, m):
            p, v, lg = e.evaluate_host(boards, want_logits=True, form=f)
            rp, rv, rlg = e.evaluate_host(S.transform(boards, f), want_logits=True)
            assert np.array_equal(p, S.unmap(rp, n, m, f)), (count, f)
            assert np.array_equal(lg, S.unmap(rlg, n, m, f)), (count, f)
            assert np.array_equal(v, rv), (count, f)
            per_form.append((p, v))
        p0, v0, lg0 = e.evaluate_host(boards, want_logits=True)
        assert np.array_equal(per_form[0][0], p0) and np.array_equal(per_form[0][1], v0)
        pa, va = e.evaluate_host(boards, form="average")
        assert np.array_equal(pa, S.average([p for p, _ in per_form])), count
        assert np.array_equal(va, S.average([v for _, v in per_form])), count
    with pytest.raises(ValueError):
        e.evaluate_host(boards[:1], form=8)
    if n != m:
        import yinyang_game_alphazero_b200 as pkg
        with pytest.raises(pkg.YinYangError):
            e.evaluate_host(boards[:1], form=1)          # rot90 changes the board's shape
    e.close()


@pytest.mark.parametrize("n,m", [(8, 8), (5, 7)])
def test_engine_modes_evaluate_like_the_forms(eng, oracle_mod, n, m):
    """yy_evaluate on a "random" engine is every board in its hashed form; on an "average" engine the averaged
    evaluation; the stub evaluator refuses the option."""
    sd = _net(n, m, 64, 2, seed=5)
    boards = _batch(oracle_mod, n, m, 300, seed=9)
    plain = eng.Engine(rows=n, cols=m, n_games=300, n_sims=1, evaluator="nn", state_dict=sd, replay_capacity=1)
    rnd = eng.Engine(rows=n, cols=m, n_games=300, n_sims=1, evaluator="nn", state_dict=sd, replay_capacity=1,
                     eval_symmetry="random", seed=1234)
    avg = eng.Engine(rows=n, cols=m, n_games=300, n_sims=1, evaluator="nn", state_dict=sd, replay_capacity=1,
                     eval_symmetry="average")
    p, v = rnd.evaluate_host(boards)
    forms = np.array([S.hashed_form(b, n, m, 1234) for b in boards])
    assert len(set(forms.tolist())) == len(S.forms(n, m))
    for f in S.forms(n, m):
        sel = forms == f
        pf, vf = plain.evaluate_host(boards[sel], form=f)
        assert np.array_equal(p[sel], pf) and np.array_equal(v[sel], vf), f
    pa, va = avg.evaluate_host(boards)
    pr, vr = plain.evaluate_host(boards, form="average")
    assert np.array_equal(pa, pr) and np.array_equal(va, vr)
    for e in (plain, rnd, avg):
        e.close()
    with pytest.raises(ValueError):
        eng.Engine(rows=n, cols=m, n_games=4, n_sims=8, evaluator="stub", eval_symmetry="random")


@pytest.mark.parametrize("step_kernels", [False, True])
@pytest.mark.parametrize("sym", ["random", "average"])
@pytest.mark.parametrize("n,m,sims", [(8, 8, 48), (6, 6, 40), (5, 7, 40)])
def test_symmetric_search_matches_oracle(eng, oracle_mod, host_tower_lib, sms, n, m, sims, sym, step_kernels):
    """A network-driven search with eval_symmetry "random" / "average" (persistent kernel, and one launch per step)
    against the oracle's search driven by the kernel's own evaluate_form in the hashed form / averaged: visit counts and
    child value sums bit for bit."""
    channels, blocks = next((c, b) for r, q, c, b in X.REPRESENTATIVES if (r, q) == (n, m))
    gb = X.tower_classes(host_tower_lib, n, m)["Gb"]
    games = sms * (gb + 1) + 5 if sym == "random" else 2 * sms + 5
    seed = 0x9E3779B97F4A7C15
    sd = _net(n, m, channels, blocks, seed=3)
    boards, players = random_play_boards(oracle_mod, n, m, games, seed=40 + n, max_frac=0.6)
    e = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="nn", state_dict=sd, cpuct=1.25,
                   step_kernels=step_kernels, eval_symmetry=sym, seed=seed)
    counts, cw = e.search_host(boards, players)
    assert e.stats().overflow == 0
    e.close()
    ev = eng.Engine(rows=n, cols=m, n_games=1, n_sims=1, evaluator="nn", state_dict=sd, replay_capacity=1,
                    eval_symmetry="average")
    cache = {}

    def predict(board):
        key = board.tobytes()
        if key not in cache:
            form = S.hashed_form(board, n, m, seed) if sym == "random" else "average"
            p, v = ev.evaluate_host(board[None], form=form)
            cache[key] = (p[0], v[0])
        return cache[key]
    for i in range(0, games, games // 9):
        r = oracle_mod.mcts_search(boards[i], int(players[i]), n, m, sims, cpuct=1.25, evaluator=predict)
        assert np.array_equal(counts[i], r["counts"]), i
        assert np.array_equal(cw[i], r["child_w"]), i
    ev.close()


def _games_by_serial(rp):
    games = {}
    for i in np.lexsort((rp["ply"], rp["game_serial"])):
        games.setdefault(int(rp["game_serial"][i]), []).append(
            (int(rp["ply"][i]), rp["boards"][i].tobytes(), rp["counts"][i].tobytes(), int(rp["player"][i]), float(rp["z"][i])))
    return games


def test_random_form_rolling_selfplay_is_reproducible(eng):
    """Rolling self-play with eval_symmetry="random": two runs with the same seed leave identical replay rings (every
    game by serial: positions, visit counts, movers, results); "none" is the default's run, and differs from it."""
    n = m = 6
    total, sims = 40, 30
    sd = _net(n, m, 128, 1, seed=11)
    runs = {}
    for tag, kw in (("random", {"eval_symmetry": "random"}), ("random2", {"eval_symmetry": "random"}),
                    ("none", {"eval_symmetry": "none"}), ("default", {})):
        e = eng.Engine(rows=n, cols=m, n_games=8, n_sims=sims, evaluator="nn", state_dict=sd, seed=77,
                       replay_capacity=total * 400, **kw)
        e.selfplay_set_quota(total)
        for _ in range(4000):
            e.selfplay_advance(97)
            st = e.stats()
            if st.games_finished >= total:
                break
        assert st.games_finished == total and st.overflow == 0
        runs[tag] = _games_by_serial(e.replay())
        e.close()
    assert sorted(runs["random"]) == list(range(total))
    assert runs["random"] == runs["random2"]
    assert runs["none"] == runs["default"]
    assert runs["random"] != runs["none"]
