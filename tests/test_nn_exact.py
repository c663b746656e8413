"""The bf16 network kernel on integer-valued networks (tests/exact_net.py), where bf16 rounding is the identity and fp32
accumulation is exact: the logits must equal the float64 reference bit for bit at every geometry class of the kernel
(position layout, FC-head tiling, clamped group size), any depth and width, and every run / group / heads-batch edge of
the persistent kernel's walk.  Also network-driven searches against the oracle, and the clean refusal of the boards the
rules accept but the network kernel does not."""
import numpy as np
import pytest

import exact_net as X
from conftest import random_play_boards

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng(yy):
    from yinyang_game_alphazero_b200 import engine
    return engine


@pytest.fixture(scope="module")
def sms(yy):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _check_batch(n, m, net, pos, out):
    """outputs of a batch whose board i is distinct position pos[i] against the float64 reference"""
    policy, value, logits = out
    A = n * m
    assert np.array_equal(logits, net.logits.astype(np.float32)[pos]), "logits differ from the exact reference"
    assert X.ulp_distance(value, np.tanh(net.pre_value).astype(np.float32)[pos]).max() <= 2, "value"
    p64 = X.softmax64(net.logits)[pos]
    normal = p64 >= 1e-30                     # exp(logit - max) stays a normal float32
    rel = np.abs(policy[normal] - p64[normal]) / p64[normal]
    assert rel.max() <= (A + 8) * 2.0 ** -24, rel.max()
    assert np.all(policy[~normal] <= 2e-30)
    first = np.full(len(net.logits), -1)
    for i, k in enumerate(pos):
        if first[k] < 0:
            first[k] = i
    assert np.array_equal(policy, policy[first[pos]]) and np.array_equal(value, value[first[pos]]), "replicas differ"


@pytest.mark.parametrize("n,m,channels,blocks", X.REPRESENTATIVES)
def test_network_is_bit_exact_on_integer_networks(eng, oracle_mod, host_tower_lib, sms, n, m, channels, blocks):
    """Per-CTA run lengths r in {1, Gb-1, Gb, Gb+1, batch, batch+1, 2 batch + Gb - 1} at count = r S and r S - 1
    (S = SM count): full groups, partial last groups of every tile count (skewed and unskewed), several heads batches per
    CTA and a trailing short CTA pair; and a batch larger than the engine, which engine_forward walks in chunks."""
    geo = X.tower_classes(host_tower_lib, n, m)
    gb, batch = geo["Gb"], geo["batch"]
    boards = X.positions(oracle_mod, n, m, 128, seed=n * 100 + m)
    net = X.ExactNet(n, m, channels, blocks, seed=1000 + n * 100 + m, boards=boards, device="cuda")
    runs = sorted({r for r in (1, gb - 1, gb, gb + 1, batch, batch + 1, 2 * batch + gb - 1) if r >= 1})
    counts = sorted({c for r in runs for c in (r * sms, r * sms - 1)})
    rng = np.random.default_rng(n * 1000 + m)
    e = eng.Engine(rows=n, cols=m, n_games=counts[-1], n_sims=1, evaluator="nn", state_dict=net.state_dict, replay_capacity=1)
    for count in counts:
        pos = rng.permutation(np.resize(np.arange(len(boards)), count))
        _check_batch(n, m, net, pos, e.evaluate_host(boards[pos], want_logits=True))
    e.close()
    small = eng.Engine(rows=n, cols=m, n_games=sms + 1, n_sims=1, evaluator="nn", state_dict=net.state_dict, replay_capacity=1)
    pos = rng.permutation(np.resize(np.arange(len(boards)), 3 * sms + 7))
    _check_batch(n, m, net, pos, small.evaluate_host(boards[pos], want_logits=True))
    small.close()


@pytest.mark.parametrize("step_kernels", [False, True])
@pytest.mark.parametrize("n,m,sims", [(10, 8, 40), (12, 12, 32), (7, 7, 48), (3, 3, 24), (32, 8, 24), (6, 6, 48)])
def test_network_search_matches_oracle(eng, oracle_mod, host_tower_lib, sms, n, m, sims, step_kernels):
    """A network-driven search (persistent kernel, and one launch per step) against the oracle's search driven by the
    kernel's own batched forward (yy_evaluate) for every board it asks about: visit counts and child value sums bit for
    bit.  More games than SMs x group size, so that some CTAs walk several groups per step."""
    channels, blocks = next((c, b) for r, q, c, b in X.REPRESENTATIVES if (r, q) == (n, m))
    gb = X.tower_classes(host_tower_lib, n, m)["Gb"]
    games = sms * (gb + 1) + 5
    net = X.ExactNet(n, m, channels, blocks, seed=7, boards=X.positions(oracle_mod, n, m, 16, seed=3), device="cuda")
    boards, players = random_play_boards(oracle_mod, n, m, games, seed=40 + n, max_frac=0.6)
    e = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="nn", state_dict=net.state_dict, cpuct=1.25,
                   step_kernels=step_kernels)
    counts, cw = e.search_host(boards, players)
    assert e.stats().overflow == 0
    e.close()
    ev = eng.Engine(rows=n, cols=m, n_games=1, n_sims=1, evaluator="nn", state_dict=net.state_dict, replay_capacity=1)
    cache = {}

    def predict(board):
        key = board.tobytes()
        if key not in cache:
            p, v = ev.evaluate_host(board[None])
            cache[key] = (p[0], v[0])
        return cache[key]
    for i in range(0, games, games // 9):
        r = oracle_mod.mcts_search(boards[i], int(players[i]), n, m, sims, cpuct=1.25, evaluator=predict)
        assert np.array_equal(counts[i], r["counts"]), i
        assert np.array_equal(cw[i], r["child_w"]), i
    ev.close()


@pytest.mark.parametrize("n,m", [(8, 23), (1, 32), (2, 30)])
def test_network_refuses_boards_wider_than_the_tower_padding(eng, oracle_mod, yy, n, m):
    """The rules take 23 <= cols <= 32, the network kernel does not (cols + 2 <= TW_PAD): an "nn" engine fails at
    creation with YinYangError, a stub engine of the same size still searches like the oracle.  (8 x 22, the widest
    board the kernel takes, is one of the representatives above.)"""
    from oracle import port
    with pytest.raises(yy.YinYangError):
        eng.Engine(rows=n, cols=m, n_games=4, n_sims=8, evaluator="nn", state_dict=port.build_net(n, m, 32, 1).state_dict())
    boards, players = random_play_boards(oracle_mod, n, m, 4, seed=n + m)
    e = eng.Engine(rows=n, cols=m, n_games=4, n_sims=40, evaluator="stub")
    counts, cw = e.search_host(boards, players)
    e.close()
    for i in range(4):
        r = oracle_mod.mcts_search(boards[i], int(players[i]), n, m, 40)
        assert np.array_equal(counts[i], r["counts"]) and np.array_equal(cw[i], r["child_w"])
