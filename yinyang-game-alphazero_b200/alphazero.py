"""Host-side mirror of the outer loop, ``AlphaZero`` (src/yin_yang/ai/alphazero.py:21-270): per iteration self-play with the
best model -> train the current model on the data directory -> evaluate current vs best -> promote at a win ratio >= 0.6.
Every stage runs on the GPU: batched self-play (self_play.generate_self_play_data), the CUDA learner
(training_pipeline.run_training_pipeline) and the batched arena (arena.evaluate).

Multi-GPU (one process per GPU under ``torchrun``, the counterpart of the reference's ``--workers`` processes): with an
initialised ``torch.distributed`` group every rank self-plays ``num_episodes / world`` games into its own data file, all
ranks train data-parallel on the shared data directory (the learner averages gradients with one all-reduce per step, so
the weights stay identical), rank 0 writes the checkpoints, plays the arena and decides the promotion."""
from __future__ import annotations

import logging
import os
import shutil

from . import arena
from .network import YinYangNeuralNetwork
from .self_play import generate_self_play_data
from .training_pipeline import run_training_pipeline

logger = logging.getLogger("YinYangAlphaZero")


def _dist():
    """(rank, world) of the initialised process group, (0, 1) without one."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except Exception:
        pass
    return 0, 1


def _barrier():
    if _dist()[1] > 1:
        import torch.distributed as dist
        dist.barrier()


class AlphaZero:
    def __init__(self, game, model_dir="models", data_dir="data", num_iterations=100, num_episodes=100, num_simulations=800,
                 num_epochs=10, temperature_threshold=10, update_threshold=0.6, num_workers=1, mcts_threads=1, eval_games=40,
                 batch_size=64, lr=0.001, eval_symmetry="none", full_search_prob=1.0, fast_simulations=None,
                 arena_opening_plies=0):
        self.game, self.model_dir, self.data_dir = game, model_dir, data_dir
        self.eval_symmetry = eval_symmetry      # leaf evaluation of the self-play and arena searches (Engine(eval_symmetry=))
        # playout cap randomisation of self-play (RollingSelfPlay); the arena always searches with num_simulations
        self.full_search_prob, self.fast_simulations = full_search_prob, fast_simulations
        self.arena_opening_plies = arena_opening_plies     # > 0: arena games start from paired random openings
        self._arena_round = 0                             # seeds the openings: every evaluation plays fresh ones
        self.num_iterations, self.num_episodes, self.num_simulations = num_iterations, num_episodes, num_simulations
        self.num_epochs, self.temperature_threshold, self.update_threshold = num_epochs, temperature_threshold, update_threshold
        self.num_workers, self.mcts_threads, self.eval_games = num_workers, mcts_threads, eval_games
        self.batch_size, self.lr = batch_size, lr
        for d in (model_dir, data_dir):
            os.makedirs(d, exist_ok=True)
        self.current_model_path = os.path.join(model_dir, "current_model.pth.tar")
        self.best_model_path = os.path.join(model_dir, "best_model.pth.tar")
        self.rank, self.world = _dist()
        if self.rank == 0:
            if not os.path.exists(self.current_model_path):
                YinYangNeuralNetwork(game).save_model(self.current_model_path)      # alphazero.py:79-83
            if not os.path.exists(self.best_model_path):
                shutil.copy(self.current_model_path, self.best_model_path)
        _barrier()

    def self_play(self, model_path):  # alphazero.py:85-108; every rank plays its share of the episodes into its own file
        from .distributed import shard_games
        lo, hi = shard_games(self.num_episodes, self.world, self.rank)
        path = generate_self_play_data(game=self.game, model_path=model_path, output_dir=self.data_dir, num_games=max(1, hi - lo),
                                       num_workers=self.num_workers, num_simulations=self.num_simulations,
                                       file_tag=f"_r{self.rank}" if self.world > 1 else "", eval_symmetry=self.eval_symmetry,
                                       full_search_prob=self.full_search_prob, fast_simulations=self.fast_simulations)
        _barrier()                                                                  # all data files are on disk
        return path

    def train(self):  # alphazero.py:110-134: one pipeline iteration over everything in data_dir, checkpoint -> current model
        new_model_path = run_training_pipeline(game=self.game, model_dir=self.model_dir, data_dir=self.data_dir, num_iterations=1,
                                               sample_size=10000, checkpoint_interval=1, epochs_per_iteration=self.num_epochs,
                                               batch_size=self.batch_size, lr=self.lr)
        if self.rank == 0:
            shutil.copy(new_model_path, self.current_model_path)
        _barrier()
        return self.current_model_path

    def evaluate(self, current_model_path, best_model_path, num_games=None):  # alphazero.py:136-226
        self._arena_round += 1
        return arena.evaluate(self.game, current_model_path, best_model_path, num_games=num_games or self.eval_games,
                              num_simulations=self.num_simulations, mcts_threads=self.mcts_threads, eval_symmetry=self.eval_symmetry,
                              opening_plies=self.arena_opening_plies, seed=self._arena_round)

    def update_best_model(self, win_ratio):  # alphazero.py:228-246
        if arena.should_promote(win_ratio, self.update_threshold):
            if self.rank == 0:
                shutil.copy(self.current_model_path, self.best_model_path)
            logger.info(f"Updated best model with win ratio {win_ratio:.2f} >= {self.update_threshold}")
            return True
        logger.info(f"Kept best model with win ratio {win_ratio:.2f} < {self.update_threshold}")
        return False

    def run_device_resident(self, slots=4096, exact_episodes=False):
        """The same loop with every example staying on the GPU(s) between self-play and the learner (device_loop.DeviceLoop):
        replay ring -> NCCL all-gather -> device replay buffer -> augmentation kernel -> learner -> NCCL weight broadcast.
        Starts from best_model.pth.tar, writes current / best / checkpoint files as a side product (rank 0)."""
        from .device_loop import DeviceLoop
        from .network import safe_load
        sd = safe_load(self.best_model_path)["state_dict"]
        from . import weights as _weights
        C, B = _weights.infer_arch(sd)
        loop = DeviceLoop(self.game, model_dir=self.model_dir, num_iterations=self.num_iterations, num_episodes=self.num_episodes,
                          num_simulations=self.num_simulations, num_epochs=self.num_epochs, batch_size=self.batch_size, lr=self.lr,
                          update_threshold=self.update_threshold, eval_games=self.eval_games, num_channels=C, num_res_blocks=B,
                          slots=slots, temperature_threshold=self.temperature_threshold, exact_episodes=exact_episodes,
                          mcts_threads=self.mcts_threads, state_dict=sd, eval_symmetry=self.eval_symmetry,
                          full_search_prob=self.full_search_prob, fast_simulations=self.fast_simulations,
                          arena_opening_plies=self.arena_opening_plies)
        try:
            return loop.run()
        finally:
            loop.close()

    def run(self):  # alphazero.py:248-270
        for iteration in range(self.num_iterations):
            logger.info(f"Starting iteration {iteration + 1}/{self.num_iterations}")
            self.self_play(self.best_model_path)
            self.train()
            win_ratio = self.evaluate(self.current_model_path, self.best_model_path) if self.rank == 0 else 0.0
            if self.world > 1:                                                      # rank 0 played the arena; everyone takes its verdict
                import torch
                import torch.distributed as dist
                t = torch.tensor([win_ratio], dtype=torch.float64, device="cuda")
                dist.broadcast(t, 0)
                win_ratio = float(t.item())
            self.update_best_model(win_ratio)
            _barrier()
            logger.info(f"Completed iteration {iteration + 1}/{self.num_iterations}")
