"""Host-side mirror of YinYangNeuralNetwork (src/yin_yang/ai/neural_network.py) for the self-play path.

The reference's network is a torch ``nn.Module`` that self-play only ever uses through ``predict(board)``
(neural_network.py:125-154) and ``load_model`` / ``save_model`` (:198-237).  Here the parameters live in a
parameter-only module with the SAME construction order and state_dict keys (so ``torch.manual_seed(s)``
yields the reference's random initialisation and reference checkpoints load unchanged), and ``predict`` runs
on the GPU: BatchNorm folded, bf16 tcgen05 tower + heads (csrc/yy_nn.cu).  There is no torch forward here.
"""
from __future__ import annotations

import os

import numpy as np
import torch
import torch.nn as nn

from . import engine as _engine


class _Block(nn.Module):  # parameter layout of ResidualBlock, neural_network.py:16-24
    def __init__(self, c):
        super().__init__()
        self.conv1 = nn.Conv2d(c, c, kernel_size=3, padding=1)
        self.bn1 = nn.BatchNorm2d(c)
        self.conv2 = nn.Conv2d(c, c, kernel_size=3, padding=1)
        self.bn2 = nn.BatchNorm2d(c)


class _Params(nn.Module):  # parameter layout + initialisation of neural_network.py:39-92
    def __init__(self, rows, cols, channels, blocks):
        super().__init__()
        A = rows * cols
        self.conv1 = nn.Conv2d(5, channels, kernel_size=3, padding=1)
        self.bn1 = nn.BatchNorm2d(channels)
        self.res_blocks = nn.ModuleList([_Block(channels) for _ in range(blocks)])
        self.policy_conv = nn.Conv2d(channels, 32, kernel_size=1)
        self.policy_bn = nn.BatchNorm2d(32)
        self.policy_fc = nn.Linear(32 * A, A)
        self.value_conv = nn.Conv2d(channels, 32, kernel_size=1)
        self.value_bn = nn.BatchNorm2d(32)
        self.value_fc1 = nn.Linear(32 * A, 256)
        self.value_fc2 = nn.Linear(256, 1)
        for mod in self.modules():
            if isinstance(mod, (nn.Conv2d, nn.Linear)):
                nn.init.xavier_normal_(mod.weight)
                if mod.bias is not None:
                    nn.init.zeros_(mod.bias)


def safe_load(filename):
    """torch.load restricted to tensors and plain containers (weights_only=True, the default of torch >= 2.6 that the
    reference's torch.load(filename, map_location='cpu') gets): a checkpoint holds a state_dict, a tuple and an int."""
    return torch.load(filename, map_location="cpu", weights_only=True)


class YinYangNeuralNetwork:
    """Drop-in for the evaluator role of the reference class: predict / load_model / save_model."""

    def __init__(self, game, num_channels=128, num_res_blocks=10, eval_symmetry="none"):
        self.game = game
        self.eval_symmetry = eval_symmetry     # predict(): "none", "random" (hashed form) or "average" (Engine(eval_symmetry=))
        self.board_size = game.getBoardSize()
        self.action_size = game.getActionSize()
        self.input_channels = 5
        self.num_channels, self.num_res_blocks = num_channels, num_res_blocks
        self._params = _Params(self.board_size[0], self.board_size[1], num_channels, num_res_blocks)
        self._engine = None
        self.weights_version = 0           # bumped whenever the parameters change: holders of device copies re-upload

    # -- parameters
    def state_dict(self):
        return self._params.state_dict()

    def load_state_dict(self, sd):
        self._params.load_state_dict(sd)
        self.weights_version += 1
        if self._engine is not None:
            self._engine.load_state_dict(self._params.state_dict())

    def save_model(self, filename):  # neural_network.py:198-215
        directory = os.path.dirname(filename)
        if directory and not os.path.exists(directory):
            os.makedirs(directory)
        torch.save({"state_dict": self.state_dict(), "board_size": self.board_size, "action_size": self.action_size},
                   filename)

    def load_model(self, filename):  # neural_network.py:217-237
        if not os.path.exists(filename):
            raise FileNotFoundError(f"Model file {filename} not found")
        ck = safe_load(filename)
        self.load_state_dict(ck["state_dict"])

    # -- inference (GPU)
    def engine(self, n_games=1):
        if self._engine is None or self._engine.n_games < n_games:
            if self._engine is not None:
                self._engine.close()
            n, m = self.board_size
            self._engine = _engine.Engine(rows=n, cols=m, n_games=n_games, n_sims=1, evaluator="nn",
                                          state_dict=self.state_dict(), rule_flags=getattr(self.game, "rule_flags", 0),
                                          eval_symmetry=self.eval_symmetry)
        return self._engine

    def predict(self, board):  # neural_network.py:125-154 -> (float32[A] softmax over ALL actions, np.float32)
        grid = board.get_board() if hasattr(board, "get_board") else np.asarray(board)
        p, v = self.engine(1).evaluate_host(np.asarray(grid, np.int8)[None])
        return p[0], np.float32(v[0])

    def predict_batch(self, grids):
        grids = np.asarray(grids, np.int8)
        return self.engine(max(1, grids.shape[0])).evaluate_host(grids)


class HashStubEvaluator:
    """Deterministic-prior evaluator (dyadic hash priors/values computed on the GPU): the mode in which visit
    counts are bit-exact against the reference (tests/golden/mcts_*.npz)."""

    def __init__(self, game):
        self.game = game
        n, m = game.getBoardSize()
        self._engine = _engine.Engine(rows=n, cols=m, n_games=1, n_sims=1, evaluator="stub")

    def predict(self, board):
        grid = board.get_board() if hasattr(board, "get_board") else np.asarray(board)
        p, v = self._engine.evaluate_host(np.asarray(grid, np.int8)[None])
        return p[0], np.float32(v[0])
