"""Model-vs-model evaluation, batched: mirror of ``AlphaZero.evaluate`` (src/yin_yang/ai/alphazero.py:136-226).

The reference plays ``num_games`` games one after the other, alternating which model moves first, every move an
``MCTS.select_action(board, player, temperature=0)``; here all games advance in lock-step and each ply costs two batched
searches (one per model, over the games in which that model is to move).  Same accounting as the reference, quirks
included: the result returned by ``getGameEnded(board, player)`` after the last move (``player`` = side to move next)
is read as "+1: the FIRST player won, -1: the second player won, anything else a draw" (alphazero.py:206-219), and the
win ratio is ``current_wins / num_games`` (:222).
"""
from __future__ import annotations

import logging

import numpy as np

from . import engine as _engine
from .mcts import MCTS
from .network import YinYangNeuralNetwork

logger = logging.getLogger("YinYangAlphaZero")


def _best_actions(mcts: MCTS, boards, players, slots):
    """select_action(..., temperature=0) for a batch: argmax of the visit distribution, lowest action on ties; a root
    without children yields the uniform distribution whose argmax is action 0 (mcts.py:183-215, 427-479)."""
    if boards.shape[0] == 0:
        return np.zeros(0, np.int32)
    pad = slots - boards.shape[0]                        # one engine size per arena: pad with empty boards
    b = np.concatenate([boards, np.zeros((pad,) + boards.shape[1:], np.int8)]) if pad else boards
    p = np.concatenate([players, np.ones(pad, np.int8)]) if pad else players
    counts, _ = mcts.search_batch(b, p)
    return counts[: boards.shape[0]].argmax(axis=1).astype(np.int32)


def play_match(game, current_mcts: MCTS, best_mcts: MCTS, num_games=40):
    """Returns dict(current_wins, best_wins, draws, win_ratio, results float64[num_games], plies int32[num_games]);
    results[i] = the reference's ``game_result`` of game i (1, -1, or 0.0001 for a draw: yin_yang_game.py:101-107)."""
    n, m = game.getBoardSize()
    flags = getattr(game, "rule_flags", 0)
    G = int(num_games)
    boards = np.zeros((G, n, m), np.int8)
    players = np.ones(G, np.int8)                        # player 1 (black) starts (alphazero.py:190)
    first_is_current = (np.arange(G) % 2) == 0           # alternate the starting model (:181-188)
    alive = np.ones(G, bool)
    results = np.zeros(G, np.float64)
    plies = np.zeros(G, np.int32)
    guard = 4 * n * m + 8                                # every ply either places a stone or passes; passes cannot repeat forever
    while alive.any() and guard > 0:
        guard -= 1
        mover_is_current = (players == 1) == first_is_current
        actions = np.full(G, -1, np.int32)
        for mc, sel in ((current_mcts, alive & mover_is_current), (best_mcts, alive & ~mover_is_current)):
            idx = np.flatnonzero(sel)
            actions[idx] = _best_actions(mc, boards[idx], players[idx], G)
        nb, npl = _engine.next_state_host(boards, players, actions, n, m, flags)
        boards[alive], players[alive] = nb[alive], npl[alive]
        plies[alive] += 1
        res = _engine.ended_host(boards, players, n, m, flags)
        ended = alive & (res != 0)
        results[ended] = res[ended]
        alive &= ~ended
    first_won, second_won = results == 1, results == -1
    current_wins = int(np.sum(first_won & first_is_current) + np.sum(second_won & ~first_is_current))
    best_wins = int(np.sum(first_won & ~first_is_current) + np.sum(second_won & first_is_current))
    draws = int(G - current_wins - best_wins)
    return {"current_wins": current_wins, "best_wins": best_wins, "draws": draws, "win_ratio": current_wins / G if G else 0.0,
            "results": results, "plies": plies}


def evaluate(game, current_model_path, best_model_path, num_games=40, num_simulations=800, mcts_threads=1, eval_symmetry="none"):
    """AlphaZero.evaluate(current_model_path, best_model_path, num_games) -> win ratio of the current model."""
    logger.info(f"Evaluating {current_model_path} against {best_model_path}")
    nets = []
    for path in (current_model_path, best_model_path):
        net = YinYangNeuralNetwork(game)
        net.load_model(path)
        nets.append(net)
    cur = MCTS(game=game, neural_net=nets[0], num_simulations=num_simulations, num_threads=mcts_threads, eval_symmetry=eval_symmetry)
    best = MCTS(game=game, neural_net=nets[1], num_simulations=num_simulations, num_threads=mcts_threads, eval_symmetry=eval_symmetry)
    try:
        out = play_match(game, cur, best, num_games)
    finally:
        cur.close(); best.close()
    logger.info(f"Evaluation completed. Current model wins: {out['current_wins']}, Best model wins: {out['best_wins']}, "
                f"Draws: {out['draws']}, Win ratio: {out['win_ratio']:.2f}")
    return out["win_ratio"]


def should_promote(win_ratio, threshold=0.6):
    """AlphaZero.update_best_model (alphazero.py:228-246): the current model replaces the best one at >= 0.6."""
    return win_ratio >= threshold
