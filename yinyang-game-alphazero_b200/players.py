"""Evaluate-mode players (src/yin_yang/yin_yang_players.py:14-42, src/yin_yang/ai/alphazero.py:272-364)."""
from __future__ import annotations

import logging
import os
import random

import numpy as np

from .mcts import MCTS
from .network import YinYangNeuralNetwork

logger = logging.getLogger("AlphaZero")


class RandomPlayer:
    """Uniformly random legal move; -1 when there is none (yin_yang_players.py:14-42)."""

    def __init__(self, game, verbose=True):
        self.game, self.verbose = game, verbose

    def play(self, board, player):
        valid = np.where(self.game.getValidMoves(board, player) == 1)[0]
        if len(valid) == 0:
            return -1
        action = int(random.choice(valid))
        if self.verbose:
            x, y = self.game._action_to_coords(action)
            print(f"{'Black' if player == 1 else 'White'} plays {chr(ord('a') + y)}{x + 1}")
        return action


class AlphaZeroPlayer:
    """MCTS-backed player (alphazero.py:272-364): search as player 1 on the canonical (= identical) board,
    temperature 0, mask with the real player's legal moves, random legal fallback."""

    def __init__(self, game, model_path, num_simulations=800, num_threads=1, eval_symmetry="none"):
        self.game = game
        self.neural_net = YinYangNeuralNetwork(game, eval_symmetry=eval_symmetry)
        if os.path.exists(model_path):
            self.neural_net.load_model(model_path)
            logger.info(f"Loaded model from {model_path}")
        else:
            logger.warning(f"No model found at {model_path}, using randomly initialized model")
        self.mcts = MCTS(game=game, neural_net=self.neural_net, num_simulations=num_simulations, num_threads=num_threads,
                         eval_symmetry=eval_symmetry)
        self.root = None

    def reset(self):
        self.root = None

    def play(self, board, player):
        valid_moves = self.game.getValidMoves(board, player)
        if np.sum(valid_moves) == 0:
            return -1
        canonical = self.game.getCanonicalForm(board, player)
        action = self.mcts.select_action(canonical, 1, valid_moves=valid_moves, temperature=0)
        if valid_moves[action] != 1:
            logger.warning(f"MCTS selected invalid move {action}, selecting a random valid move instead")
            idx = np.where(valid_moves == 1)[0]
            if len(idx) == 0:
                return -1
            action = int(np.random.choice(idx))
        return int(action)

    def notify(self, board, action):
        """Tree reuse is a no-op in the reference's search path (SURVEY Q7); kept for interface parity."""
        return None
