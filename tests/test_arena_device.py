"""The device arena (yy_arena_run / arena.DeviceArena): both models' searches in one persistent-kernel launch, every game
moving between its two models' trees on the device.  It must play the very games arena.play_match plays (which
test_gpu_facade pins to the reference's sequential loop): results, plies and the counts, game for game."""
import ctypes
import os
import sys

import numpy as np
import pytest

from conftest import randomise_bn

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg(yy):
    from yinyang_game_alphazero_b200 import arena, engine, game, mcts, network, weights
    return dict(arena=arena, engine=engine, game=game, mcts=mcts, network=network, weights=weights)


def _nets(pkg, game, C, B, seeds=(1, 2)):
    import torch
    sds = []
    for s in seeds:
        torch.manual_seed(s)
        n, m = game.getBoardSize()
        net = randomise_bn(pkg["network"]._Params(n, m, C, B), seed=s)
        sds.append(net.state_dict())
    return sds


def _host_match(pkg, game, sds, C, B, sims, G, sym="none", **kw):
    """arena.play_match with one MCTS per model (the host loop the device arena must reproduce)."""
    mc = []
    for sd in sds:
        net = pkg["network"].YinYangNeuralNetwork(game, num_channels=C, num_res_blocks=B)
        net.load_state_dict(sd)
        mc.append(pkg["mcts"].MCTS(game, net, num_simulations=sims, verbose=0, eval_symmetry=sym))
    try:
        return pkg["arena"].play_match(game, mc[0], mc[1], G, **kw)
    finally:
        for m in mc:
            m.close()


def _device_match(pkg, game, sds, C, B, sims, G, sym="none", openings=None, max_plies=None):
    a = pkg["arena"].DeviceArena(game, G, sims, C, B, eval_symmetry=sym)
    try:
        return a.play(sds[0], sds[1], openings, max_plies=max_plies)
    finally:
        a.close()


def _same(d, h):
    assert np.array_equal(d["results"], h["results"]), (d["results"], h["results"])
    assert np.array_equal(d["plies"], h["plies"]), (d["plies"], h["plies"])
    for k in ("current_wins", "best_wins", "draws", "win_ratio"):
        assert d[k] == h[k], k


@pytest.mark.parametrize("n,m,C,B,sims,sym,G", [
    (5, 5, 16, 1, 16, "none", 6),
    (5, 5, 16, 1, 16, "random", 1),
    (6, 6, 32, 2, 32, "none", 17),
    (6, 6, 16, 3, 24, "average", 6),
    (8, 8, 32, 1, 16, "random", 17),
    (8, 8, 16, 2, 64, "none", 1),
    (5, 7, 16, 2, 16, "average", 17),
    (4, 6, 32, 1, 32, "random", 6),
])
def test_device_arena_equals_play_match(pkg, n, m, C, B, sims, sym, G):
    game = pkg["game"].YinYangGame(n, m)
    sds = _nets(pkg, game, C, B)
    h = _host_match(pkg, game, sds, C, B, sims, G, sym)
    d = _device_match(pkg, game, sds, C, B, sims, G, sym)
    _same(d, h)
    assert np.all(d["plies"] > 0)


@pytest.mark.parametrize("n,m,plies,G", [(6, 6, 2, 8), (5, 7, 6, 7), (8, 8, 6, 6)])
def test_openings_equal_play_match(pkg, n, m, plies, G):
    game = pkg["game"].YinYangGame(n, m)
    sds = _nets(pkg, game, 16, 1, seeds=(3, 4))
    op = pkg["arena"].make_openings(game, G, plies, seed=11)
    h = _host_match(pkg, game, sds, 16, 1, 16, G, openings=op)
    d = _device_match(pkg, game, sds, 16, 1, 16, G, openings=op)
    _same(d, h)
    # pair i = one opening, the colours swapped
    assert np.array_equal(op["black"][0::2][: G // 2], op["black"][1::2][: G // 2])
    assert list(op["a_plays_black"][:4]) == [True, False, True, False]


def test_openings_already_over(pkg):
    """A 4x4 opening that is terminal before the first move gives a 0-ply game, on the device as in play_match."""
    import torch
    game = pkg["game"].YinYangGame(4, 4)
    eng = pkg["engine"]
    G, plies = 8, 14
    for seed in range(64):
        op = pkg["arena"].make_openings(game, G, plies, seed)
        code = eng.ended(torch.from_numpy(op["black"].view(np.int64)).cuda(), torch.from_numpy(op["white"].view(np.int64)).cuda(),
                         torch.from_numpy(op["player"]).cuda(), 4, 4).cpu().numpy()
        if (code != 0).any() and (code == 0).any():
            break
    else:
        pytest.fail("no 4x4 opening seed with both terminal and live starts")
    sds = _nets(pkg, game, 16, 1)
    h = _host_match(pkg, game, sds, 16, 1, 16, G, openings=op)
    d = _device_match(pkg, game, sds, 16, 1, 16, G, openings=op)
    _same(d, h)
    assert np.array_equal(d["plies"] == 0, code != 0)


def test_games_do_not_depend_on_the_slot(pkg):
    game = pkg["game"].YinYangGame(6, 6)
    sds = _nets(pkg, game, 16, 2)
    op = pkg["arena"].make_openings(game, 9, 4, seed=5)
    sub = pkg["arena"].shard_openings
    full = _device_match(pkg, game, sds, 16, 2, 16, 9, openings=op)
    part = _device_match(pkg, game, sds, 16, 2, 16, 4, openings=sub(op, 4, 8))
    assert np.array_equal(part["results"], full["results"][4:8]) and np.array_equal(part["plies"], full["plies"][4:8])
    for i in (0, 7):
        one = _device_match(pkg, game, sds, 16, 2, 16, 1, openings=sub(op, i, i + 1))
        assert one["results"][0] == full["results"][i] and one["plies"][0] == full["plies"][i]


def test_ply_cap(pkg):
    game = pkg["game"].YinYangGame(6, 6)
    sds = _nets(pkg, game, 16, 1)
    cap = 7
    h = _host_match(pkg, game, sds, 16, 1, 16, 6, max_plies=cap)
    d = _device_match(pkg, game, sds, 16, 1, 16, 6, max_plies=cap)
    _same(d, h)
    capped = d["plies"] == cap
    assert capped.any() and np.all(d["results"][capped] == 0) and np.all(d["plies"] <= cap)


def _raw_arena(eng, image, nbytes, G=1, max_plies=10):
    import torch
    L, W, dev = eng.L, eng.W, eng.tdev
    b = torch.zeros((G, W), dtype=torch.int64, device=dev)
    p = torch.ones(G, dtype=torch.int8, device=dev)
    ab = torch.ones(G, dtype=torch.uint8, device=dev)
    code = torch.zeros(G, dtype=torch.int8, device=dev)
    plies = torch.zeros(G, dtype=torch.int32, device=dev)
    P = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    return L.yy_arena_run(eng.handle, P(image), nbytes, P(b), P(b), P(p), P(ab), max_plies, P(code), P(plies), None)


def test_refusals(pkg):
    E = pkg["engine"]
    game = pkg["game"].YinYangGame(5, 5)
    sd = _nets(pkg, game, 16, 1, seeds=(1,))[0]
    kw = dict(rows=5, cols=5, n_sims=8, state_dict=sd)
    ok = E.Engine(n_games=2, evaluator="nn", **kw)
    img, nb = ok.weight_image, ok.weight_image.numel()
    assert _raw_arena(ok, img, nb) == 0
    assert _raw_arena(ok, img, nb - 1) == -1                                 # YY_ERR_INVALID: wrong image size
    assert _raw_arena(ok, img, nb, max_plies=0) == -1                        # YY_ERR_INVALID: max_plies < 1
    odd = E.Engine(n_games=3, evaluator="nn", **kw)
    assert _raw_arena(odd, img, nb) == -1                                    # YY_ERR_INVALID: odd n_games
    for eng in (E.Engine(rows=5, cols=5, n_games=2, n_sims=8, evaluator="stub"),
                E.Engine(rows=5, cols=5, n_games=2, n_sims=8, evaluator="external"),
                E.Engine(n_games=2, evaluator="nn", leaves_per_step=2, **kw),
                E.Engine(n_games=2, evaluator="nn", step_kernels=True, **kw)):
        assert _raw_arena(eng, img, nb) == -5                                # YY_ERR_STATE
        eng.close()
    with pytest.raises(E._lib.YinYangError):
        import torch
        odd.arena_run(img, torch.zeros((1, 1), dtype=torch.int64, device="cuda"), torch.zeros((1, 1), dtype=torch.int64, device="cuda"),
                      torch.ones(1, dtype=torch.int8, device="cuda"), torch.ones(1, dtype=torch.uint8, device="cuda"), 10)
    ok.close(); odd.close()


def test_device_loop_arena_equals_play_match(pkg):
    from yinyang_game_alphazero_b200.device_loop import DeviceLoop
    game = pkg["game"].YinYangGame(6, 6)
    loop = DeviceLoop(game, num_iterations=1, num_episodes=8, num_simulations=16, num_epochs=1, batch_size=32, sample_size=128,
                      eval_games=6, num_channels=16, num_res_blocks=1, slots=8, save_files=False, seed=1)
    try:
        best0 = loop.best_sd
        out = loop.run_iteration(0)
        cur = loop.learner.state_dict()
    finally:
        loop.close()
    h = _host_match(pkg, game, [cur, best0], 16, 1, 16, 6)
    assert out["win_ratio"] == h["win_ratio"]


def test_train_cli_with_openings(tmp_path):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    md, dd = str(tmp_path / "models"), str(tmp_path / "data")
    r = subprocess.run([sys.executable, os.path.join(root, "train_alphazero.py"), "--mode", "train", "--rows", "6", "--cols", "6",
                        "--iterations", "1", "--episodes", "8", "--simulations", "16", "--epochs", "1", "--arena-games", "6",
                        "--arena-opening-plies", "4", "--model-dir", md, "--data-dir", dd],
                       capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
