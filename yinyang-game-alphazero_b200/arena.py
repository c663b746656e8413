"""Model-vs-model evaluation, batched: mirror of ``AlphaZero.evaluate`` (src/yin_yang/ai/alphazero.py:136-226).

The reference plays ``num_games`` games one after the other, alternating which model moves first, every move an
``MCTS.select_action(board, player, temperature=0)``; here all games advance in lock-step and each ply costs two batched
searches (one per model, over the games in which that model is to move).  Same accounting as the reference, quirks
included: the result returned by ``getGameEnded(board, player)`` after the last move (``player`` = side to move next)
is read as "+1: the FIRST player won, -1: the second player won, anything else a draw" (alphazero.py:206-219), and the
win ratio is ``current_wins / num_games`` (:222).

``DeviceArena`` plays the same games on the persistent search kernel: both models in one launch, every game moving between
its two models' trees on the device (yy_arena_run), no host round trip between plies.  ``make_openings`` gives the games
paired random openings, so that they differ from one another (from the empty board, every game in which a model plays
black is the same deterministic game).
"""
from __future__ import annotations

import logging

import numpy as np

from . import bitboard, engine as _engine, weights as _weights
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


def default_max_plies(game):
    """The ply cap of play_match: every ply either places a stone or passes, and passes cannot repeat forever."""
    n, m = game.getBoardSize()
    return 4 * n * m + 8


def tally(results, a_plays_black):
    """The reference's accounting (alphazero.py:206-222): results[i] = +1 counts for the model playing black in game i,
    -1 for the one playing white, anything else is a draw.  a_plays_black[i]: the current model plays black."""
    results = np.asarray(results, np.float64)
    a_black = np.asarray(a_plays_black, bool)
    first_won, second_won = results == 1, results == -1
    current_wins = int(np.sum(first_won & a_black) + np.sum(second_won & ~a_black))
    best_wins = int(np.sum(first_won & ~a_black) + np.sum(second_won & a_black))
    G = int(results.size)
    return {"current_wins": current_wins, "best_wins": best_wins, "draws": G - current_wins - best_wins,
            "win_ratio": current_wins / G if G else 0.0}


def make_openings(game, num_games, plies, seed):
    """Start positions of an arena: games 2i and 2i + 1 start from engine.random_playout position i (``plies`` uniformly
    random legal plies, keyed by (seed, i)); the current model plays black in game 2i and white in 2i + 1 (play_match's
    colour assignment).  plies = 0: empty boards, black to move.  Opening i does not depend on num_games, so a shard of
    games [lo, hi) is the slice [lo:hi].  Returns dict(black, white uint64[G, W], player int8[G], a_plays_black bool[G])."""
    n, m = game.getBoardSize()
    G, W = int(num_games), bitboard.words_for(n, m)
    pairs = (G + 1) // 2
    if plies > 0 and pairs:
        import torch
        b, w, p = _engine.random_playout(pairs, torch.full((pairs,), int(plies), dtype=torch.int32), n, m, seed=int(seed),
                                         rule_flags=getattr(game, "rule_flags", 0))
        b, w, p = (t.cpu().numpy() for t in (b, w, p))
        b, w = b.view(np.uint64), w.view(np.uint64)
    else:
        b, w, p = np.zeros((pairs, W), np.uint64), np.zeros((pairs, W), np.uint64), np.ones(pairs, np.int8)
    idx = np.arange(G) // 2
    return {"black": np.ascontiguousarray(b[idx]), "white": np.ascontiguousarray(w[idx]), "player": np.asarray(p, np.int8)[idx],
            "a_plays_black": (np.arange(G) % 2) == 0}


def shard_openings(openings, lo, hi):
    return {k: v[lo:hi] for k, v in openings.items()}


def play_match(game, current_mcts: MCTS, best_mcts: MCTS, num_games=40, openings=None, max_plies=None):
    """Returns dict(current_wins, best_wins, draws, win_ratio, results float64[num_games], plies int32[num_games]);
    results[i] = the reference's ``game_result`` of game i (1, -1, or 0.0001 for a draw: yin_yang_game.py:101-107).
    openings (make_openings): start boards, players and colours instead of empty boards; a game whose start position is
    already over ends with 0 plies.  max_plies: the ply cap (default_max_plies); a game that reaches it scores 0."""
    n, m = game.getBoardSize()
    flags = getattr(game, "rule_flags", 0)
    G = int(num_games)
    boards = np.zeros((G, n, m), np.int8)
    players = np.ones(G, np.int8)                        # player 1 (black) starts (alphazero.py:190)
    first_is_current = (np.arange(G) % 2) == 0           # alternate the starting model (:181-188)
    alive = np.ones(G, bool)
    results = np.zeros(G, np.float64)
    plies = np.zeros(G, np.int32)
    if openings is not None:
        boards = bitboard.unpack_boards(openings["black"][:G], openings["white"][:G], n, m).astype(np.int8)
        players = np.asarray(openings["player"][:G], np.int8).copy()
        first_is_current = np.asarray(openings["a_plays_black"][:G], bool)
        res = _engine.ended_host(boards, players, n, m, flags)
        results[res != 0] = res[res != 0]
        alive &= res == 0
    guard = default_max_plies(game) if max_plies is None else int(max_plies)
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
    return {**tally(results, first_is_current), "results": results, "plies": plies}


class DeviceArena:
    """play_match for the network evaluator and mcts_threads = 1 on ONE engine of 2 x num_games slots (yy_arena_run):
    slots [0, G) search with the current model, [G, 2G) with the best one, both halves in the same launches.  Reused across
    iterations: play() only swaps the weight images.  seed = the engine seed (the form hash of eval_symmetry="random")."""

    def __init__(self, game, num_games, num_simulations=800, channels=128, blocks=10, eval_symmetry="none", seed=0, device=None):
        import torch
        self.game, self.G = game, int(num_games)
        self.n, self.m = game.getBoardSize()
        self.channels, self.blocks = int(channels), int(blocks)
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.eng = _engine.Engine(rows=self.n, cols=self.m, n_games=2 * self.G, n_sims=int(num_simulations), evaluator="nn",
                                  rule_flags=getattr(game, "rule_flags", 0), seed=seed, eval_symmetry=eval_symmetry, device=self.device,
                                  nn_channels=self.channels, nn_blocks=self.blocks, replay_capacity=1,
                                  weight_image=self._image(None))

    def _image(self, image_or_sd):
        """A packed device image (uint8 tensor, 256-byte aligned) or a state dict -> device image; None: zeros."""
        import torch
        if torch.is_tensor(image_or_sd):
            return image_or_sd
        if image_or_sd is None:
            size = int(_engine._lib.lib().yy_nn_weight_bytes(self.n, self.m, self.channels, self.blocks))
            return _engine.device_image(np.zeros(size, np.uint8), self.device)
        return _engine.device_image(_weights.pack_state_dict(image_or_sd, self.n, self.m), self.device)

    def close(self):
        self.eng.close()

    def play(self, current, best, openings=None, max_plies=None):
        """current / best: packed device images or state dicts.  Returns play_match's dict for the same games."""
        import torch
        G = self.G
        if openings is None:
            openings = make_openings(self.game, G, 0, 0)
        cur, bst = self._image(current), self._image(best)
        self.eng.load_weight_image(cur)
        dev = self.eng.tdev
        b = torch.from_numpy(np.ascontiguousarray(openings["black"][:G]).view(np.int64)).to(dev)
        w = torch.from_numpy(np.ascontiguousarray(openings["white"][:G]).view(np.int64)).to(dev)
        p = torch.from_numpy(np.ascontiguousarray(openings["player"][:G], np.int8)).to(dev)
        ab = np.asarray(openings["a_plays_black"][:G], bool)
        codes, plies = self.eng.arena_run(bst, b, w, p, torch.from_numpy(ab.astype(np.uint8)).to(dev),
                                          default_max_plies(self.game) if max_plies is None else max_plies)
        codes, plies = _engine._to_host(codes, plies)
        results = _engine.result_from_code(codes)
        return {**tally(results, ab), "results": results, "plies": plies.astype(np.int32)}


def play_sharded(num_games, play, rank=0, world=1, group=None, device="cpu"):
    """The arena's games spread over the ranks in whole pairs (distributed.shard_games over the pairs): this rank plays games
    [lo, hi) with play(lo, hi) -> dict(current_wins, best_wins, draws), and the counts are summed over the ranks, so every
    rank returns the same dict(current_wins, best_wins, draws, win_ratio)."""
    import torch
    from .distributed import shard_games
    G = int(num_games)
    plo, phi = shard_games((G + 1) // 2, world, rank)
    lo, hi = min(G, 2 * plo), min(G, 2 * phi)
    out = play(lo, hi) if hi > lo else {"current_wins": 0, "best_wins": 0, "draws": 0}
    t = torch.tensor([out["current_wins"], out["best_wins"], out["draws"]], dtype=torch.int64, device=device)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, group=group)
    cw, bw, dr = (int(x) for x in t.tolist())
    return {"current_wins": cw, "best_wins": bw, "draws": dr, "win_ratio": cw / G if G else 0.0}


def evaluate(game, current_model_path, best_model_path, num_games=40, num_simulations=800, mcts_threads=1, eval_symmetry="none",
             opening_plies=0, seed=0):
    """AlphaZero.evaluate(current_model_path, best_model_path, num_games) -> win ratio of the current model.  opening_plies > 0:
    paired random openings (make_openings(..., seed)).  mcts_threads = 1 plays on the device arena, K > 1 on the host loop."""
    logger.info(f"Evaluating {current_model_path} against {best_model_path}")
    nets = []
    for path in (current_model_path, best_model_path):
        net = YinYangNeuralNetwork(game)
        net.load_model(path)
        nets.append(net)
    openings = make_openings(game, num_games, opening_plies, seed) if opening_plies > 0 else None
    if mcts_threads == 1 and num_games > 0:
        sds = [net.state_dict() for net in nets]
        C, B = _weights.infer_arch(sds[0])
        arena = DeviceArena(game, num_games, num_simulations, C, B, eval_symmetry=eval_symmetry)
        try:
            out = arena.play(sds[0], sds[1], openings)
        finally:
            arena.close()
    else:
        cur = MCTS(game=game, neural_net=nets[0], num_simulations=num_simulations, num_threads=mcts_threads, eval_symmetry=eval_symmetry)
        best = MCTS(game=game, neural_net=nets[1], num_simulations=num_simulations, num_threads=mcts_threads, eval_symmetry=eval_symmetry)
        try:
            out = play_match(game, cur, best, num_games, openings=openings)
        finally:
            cur.close(); best.close()
    logger.info(f"Evaluation completed. Current model wins: {out['current_wins']}, Best model wins: {out['best_wins']}, "
                f"Draws: {out['draws']}, Win ratio: {out['win_ratio']:.2f}")
    return out["win_ratio"]


def should_promote(win_ratio, threshold=0.6):
    """AlphaZero.update_best_model (alphazero.py:228-246): the current model replaces the best one at >= 0.6."""
    return win_ratio >= threshold
