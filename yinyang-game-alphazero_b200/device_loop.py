"""The AlphaZero outer loop with everything between self-play and the learner resident on the GPU(s).

Mirror of ``AlphaZero.run`` (src/yin_yang/ai/alphazero.py:248-270: self-play with the best model -> train the current
model -> arena -> promote at >= 0.6) in which no example ever becomes a Python object or a file on its way to the
learner: finished games go from the engine's replay ring (device) -> NCCL all-gather over the ranks -> a device replay
buffer (the 500,000-example deque of training_pipeline.py:23-106) -> sampled records -> yy_augment_samples (8 forms) ->
Learner.step (one all-reduce of the gradients per step) -> packed weight image -> NCCL broadcast -> every rank's engine.
One process per GPU (``torchrun``); files (checkpoints, replay export) are an optional side product written by rank 0.
"""
from __future__ import annotations

import logging
import os
import time

import numpy as np
import torch

from . import engine as _engine, weights as _weights
from .learner import Learner

logger = logging.getLogger("YinYangAlphaZero")


def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist, dist.get_rank(), dist.get_world_size()
    return None, 0, 1


class DeviceReplayBuffer:
    """TrainingDataQueue (training_pipeline.py:23-106) on the device: a ring of the newest ``max_size`` examples
    (deque(maxlen) semantics), ``sample(k)`` = random.sample without replacement.  Records: bitboards, visit counts, z."""

    def __init__(self, W, A, max_size=500000, device="cuda"):
        self.cap, self.W, self.A = int(max_size), W, A
        self.black = torch.zeros((self.cap, W), dtype=torch.int64, device=device)
        self.white = torch.zeros((self.cap, W), dtype=torch.int64, device=device)
        self.counts = torch.zeros((self.cap, A), dtype=torch.int16, device=device)
        self.z = torch.zeros(self.cap, dtype=torch.float32, device=device)
        self.size, self.head = 0, 0                      # head = next slot to overwrite

    def __len__(self):
        return self.size

    def push(self, black, white, counts, z):
        n = int(z.shape[0])
        if n == 0:
            return
        if n >= self.cap:                                # only the newest cap examples survive
            black, white, counts, z, n = black[-self.cap:], white[-self.cap:], counts[-self.cap:], z[-self.cap:], self.cap
        idx = (self.head + torch.arange(n, device=self.z.device)) % self.cap
        self.black[idx], self.white[idx], self.counts[idx], self.z[idx] = black, white, counts, z
        self.head = (self.head + n) % self.cap
        self.size = min(self.cap, self.size + n)

    def sample(self, k, generator=None):
        k = min(int(k), self.size)
        idx = torch.randperm(self.size, device=self.z.device, generator=generator)[:k]
        return self.black[idx], self.white[idx], self.counts[idx], self.z[idx]


class DeviceSelfPlay:
    """Rolling self-play whose finished games stay on the device (engine replay ring -> device tensors)."""

    def __init__(self, game, state_dict, slots=4096, num_simulations=800, temperature_threshold=10, dirichlet_alpha=0.3,
                 dirichlet_epsilon=0.25, cpuct=1.0, seed=0, evaluator="nn", device=None, eval_symmetry="none", full_search_prob=1.0,
                 fast_simulations=None):
        self.n, self.m = game.getBoardSize()
        self.A, self.slots, self.sims = self.n * self.m, int(slots), int(num_simulations)
        self.eng = _engine.Engine(rows=self.n, cols=self.m, n_games=self.slots, n_sims=self.sims, evaluator=evaluator, cpuct=cpuct,
                                  rule_flags=getattr(game, "rule_flags", 0), dirichlet_alpha=dirichlet_alpha,
                                  dirichlet_epsilon=dirichlet_epsilon, temperature_threshold=temperature_threshold, seed=seed,
                                  state_dict=state_dict, replay_capacity=self.slots * (2 * self.A + 8) + 4096, device=device,
                                  eval_symmetry=eval_symmetry)
        if full_search_prob != 1.0 or fast_simulations is not None:      # playout cap: only full searches are recorded
            self.eng.selfplay_set_playout_cap(full_search_prob, fast_simulations)
        self.cursor, self._pend = 0, None
        self.games_done = 0

    def close(self):
        self.eng.close()

    def set_weight_image(self, image_u8):
        self.eng.load_weight_image(image_u8)

    def _collect(self):
        """Moves the records appended since the last call out of the ring; returns those of finished games (device)."""
        eng = self.eng
        st = eng.stats()
        if st.overflow:
            raise _engine._lib.YinYangError("a tree arena overflowed: raise edges_per_game")
        if st.examples - self.cursor > eng.replay_capacity:
            raise _engine._lib.YinYangError("replay ring overrun")
        new = {k: v.clone() for k, v in eng.replay_window_dev(self.cursor, st.examples).items()}
        self.cursor = st.examples
        if self._pend is not None:
            new = {k: torch.cat([self._pend[k], new[k]]) for k in new}
        results = eng.replay_views()["results"]
        code = results[(new["game_serial"].long() % eng.results_capacity)] if new["ply"].numel() else torch.zeros(0, dtype=torch.int8, device=results.device)
        done = code != 0
        self._pend = {k: v[~done] for k, v in new.items()}
        c = code[done].float()
        z = torch.where(c == 2, torch.full_like(c, _engine.DRAW_VALUE), c)            # yin_yang_game.py:101-107
        self.games_done = st.games_finished
        return {"black": new["black"][done], "white": new["white"][done], "counts": new["counts"][done], "z": z}

    def play(self, num_games, exact=False):
        """Advances the slots until ``num_games`` more games are finished; returns their examples (and those of every other
        game that finished meanwhile) as device tensors.  exact=False keeps the unfinished games in flight for the next call
        (no tail); exact=True starts exactly ``num_games`` games (game quota) and waits for all of them."""
        target = self.games_done + num_games
        self.eng.selfplay_set_quota(target if exact else None)
        parts, guard = [], 0
        while self.games_done < target and guard < 100000:
            self.eng.selfplay_advance(self.sims + 1)
            parts.append(self._collect())
            guard += 1
        keys = ("black", "white", "counts", "z")
        return {k: torch.cat([p[k] for p in parts]) if parts else None for k in keys}


class DeviceLoop:
    """AlphaZero.run (alphazero.py:248-270), device resident, one instance per rank."""

    def __init__(self, game, model_dir="models", num_iterations=100, num_episodes=100, num_simulations=800, num_epochs=10,
                 batch_size=64, lr=0.001, weight_decay=1e-4, sample_size=10000, queue_size=500000, update_threshold=0.6, eval_games=40,
                 num_channels=128, num_res_blocks=10, slots=4096, temperature_threshold=10, exact_episodes=False, save_files=True,
                 seed=0, mcts_threads=1, state_dict=None, eval_symmetry="none", full_search_prob=1.0, fast_simulations=None,
                 arena_opening_plies=0):
        self.game, self.model_dir = game, model_dir
        self.eval_symmetry = eval_symmetry
        self.num_iterations, self.num_episodes, self.num_simulations, self.num_epochs = num_iterations, num_episodes, num_simulations, num_epochs
        self.batch_size, self.sample_size, self.update_threshold, self.eval_games = batch_size, sample_size, update_threshold, eval_games
        self.exact_episodes, self.save_files, self.mcts_threads = exact_episodes, save_files, mcts_threads
        self.seed, self.arena_opening_plies = seed, arena_opening_plies
        self._device_arena = None
        self.dist, self.rank, self.world = _dist()
        n, m = game.getBoardSize()
        self.n, self.m = n, m
        from .network import YinYangNeuralNetwork
        if state_dict is None:
            state_dict = YinYangNeuralNetwork(game, num_channels, num_res_blocks).state_dict()      # alphazero.py:79-83
        self.learner = Learner(n, m, num_channels, num_res_blocks, batch_size=batch_size, lr=lr, weight_decay=weight_decay,
                               state_dict=state_dict, data_parallel=True)                           # adopts rank 0's weights
        self.best_sd = self.learner.state_dict()
        share = -(-num_episodes // self.world)
        self.episodes_per_rank = share
        self.selfplay = DeviceSelfPlay(game, self.best_sd, slots=max(1, min(slots, share)), num_simulations=num_simulations,
                                       temperature_threshold=temperature_threshold, seed=seed * 1000003 + self.rank,
                                       eval_symmetry=eval_symmetry, full_search_prob=full_search_prob,
                                       fast_simulations=fast_simulations)
        self.buffer = DeviceReplayBuffer(self.selfplay.eng.W, n * m, queue_size)
        self.gen = torch.Generator(device="cuda")
        self.gen.manual_seed(seed * 7919 + self.rank)
        self.history = []
        if save_files and self.rank == 0:
            os.makedirs(model_dir, exist_ok=True)

    def close(self):
        self.selfplay.close()
        if self._device_arena is not None:
            self._device_arena.close()

    # -- stages
    def _gather(self, rec):
        if self.world == 1:
            return rec
        from . import distributed as yyd
        return yyd.gather_records(rec, dst=None)

    def _train(self):
        metrics = {"policy_loss": [], "value_loss": [], "total_loss": []}
        black, white, counts, z = self.buffer.sample(self.sample_size, self.gen)
        planes, pol, val = _engine.augment_samples(black, white, self.n, self.m, counts=counts, values=z)   # 8 forms per record
        n = planes.shape[0]
        steps = 0
        for _ in range(self.num_epochs):
            perm = torch.randperm(n, device=planes.device, generator=self.gen)
            pl, po, va = planes[perm], pol[perm], val[perm]
            acc = torch.zeros(2, dtype=torch.float64, device=planes.device)
            for i in range(0, n, self.batch_size):
                j = min(n, i + self.batch_size)
                acc += self.learner.step(pl[i:j], po[i:j], va[i:j]).double() * (j - i)
                steps += 1
            p, v = (acc / max(n, 1)).tolist()
            metrics["policy_loss"].append(p); metrics["value_loss"].append(v); metrics["total_loss"].append(p + v)
        return metrics, steps

    def _broadcast_weights(self, sd):
        """rank 0 packs the network (BatchNorm folded, bf16 streams), the image goes to every engine over NCCL."""
        eng = self.selfplay.eng
        if self.rank == 0:
            img = torch.from_numpy(_weights.pack_state_dict(sd, self.n, self.m)).to(eng.weight_image.device)
            eng.weight_image.copy_(img)
        if self.world > 1:
            self.dist.broadcast(eng.weight_image, 0)
        eng.load_weight_image(eng.weight_image)

    def _arena(self, current_sd, it=0):
        """alphazero.py:136-226.  mcts_threads = 1: the device arena (arena.DeviceArena) with the current weights against the
        self-play engine's image of best_sd, the games sharded over the ranks in whole pairs and the counts all-reduced.
        Otherwise rank 0 plays the host loop and every rank takes its verdict."""
        from . import arena
        if self.mcts_threads == 1 and self.eval_games > 0:
            openings = arena.make_openings(self.game, self.eval_games, self.arena_opening_plies, self.seed * 1000003 + it)
            C, B = _weights.infer_arch(current_sd)

            def play(lo, hi):
                if self._device_arena is None or self._device_arena.G != hi - lo:
                    if self._device_arena is not None:
                        self._device_arena.close()
                    self._device_arena = arena.DeviceArena(self.game, hi - lo, self.num_simulations, C, B,
                                                           eval_symmetry=self.eval_symmetry)
                return self._device_arena.play(current_sd, self.selfplay.eng.weight_image, arena.shard_openings(openings, lo, hi))
            return arena.play_sharded(self.eval_games, play, self.rank, self.world, device="cuda")["win_ratio"]
        ratio = 0.0
        if self.rank == 0 and self.eval_games > 0:
            from . import arena
            from .mcts import MCTS
            from .network import YinYangNeuralNetwork
            C, B = _weights.infer_arch(current_sd)
            nets = []
            for sd in (current_sd, self.best_sd):
                net = YinYangNeuralNetwork(self.game, C, B)
                net.load_state_dict(sd)
                nets.append(net)
            cur = MCTS(self.game, nets[0], num_simulations=self.num_simulations, num_threads=self.mcts_threads, verbose=0,
                       eval_symmetry=self.eval_symmetry)
            best = MCTS(self.game, nets[1], num_simulations=self.num_simulations, num_threads=self.mcts_threads, verbose=0,
                        eval_symmetry=self.eval_symmetry)
            try:
                ratio = arena.play_match(self.game, cur, best, self.eval_games)["win_ratio"]
            finally:
                cur.close(); best.close()
        if self.world > 1:
            t = torch.tensor([ratio], dtype=torch.float64, device="cuda")
            self.dist.broadcast(t, 0)
            ratio = float(t.item())
        return ratio

    def run_iteration(self, it):
        sync = torch.cuda.synchronize
        t0 = time.perf_counter()
        rec = self.selfplay.play(self.episodes_per_rank, exact=self.exact_episodes)
        sync(); t1 = time.perf_counter()
        allrec = self._gather(rec)
        self.buffer.push(allrec["black"], allrec["white"], allrec["counts"], allrec["z"])
        sync(); t2 = time.perf_counter()
        metrics, steps = self._train()
        sync(); t3 = time.perf_counter()
        current_sd = self.learner.state_dict()
        ratio = self._arena(current_sd, it)
        promoted = ratio >= self.update_threshold
        t4 = time.perf_counter()
        if promoted:
            self.best_sd = current_sd
            self._broadcast_weights(self.best_sd)
        sync(); t5 = time.perf_counter()
        if self.save_files and self.rank == 0:
            from .network import YinYangNeuralNetwork
            C, B = _weights.infer_arch(current_sd)
            net = YinYangNeuralNetwork(self.game, C, B)
            net.load_state_dict(current_sd)
            net.save_model(os.path.join(self.model_dir, "current_model.pth.tar"))
            net.save_model(os.path.join(self.model_dir, f"checkpoint_{it + 1}.pth.tar"))
            if promoted or it == 0:
                net.load_state_dict(self.best_sd)
                net.save_model(os.path.join(self.model_dir, "best_model.pth.tar"))
        out = {"iteration": it + 1, "examples_local": int(rec["z"].shape[0]), "examples_global": int(allrec["z"].shape[0]),
               "buffer": len(self.buffer), "learner_steps": steps, "self_play_s": t1 - t0, "gather_s": t2 - t1, "train_s": t3 - t2,
               "arena_s": t4 - t3, "broadcast_s": t5 - t4, "win_ratio": ratio, "promoted": bool(promoted),
               "policy_loss": metrics["policy_loss"][-1] if metrics["policy_loss"] else None,
               "value_loss": metrics["value_loss"][-1] if metrics["value_loss"] else None}
        self.history.append(out)
        if self.rank == 0:
            logger.info("iteration %(iteration)d: %(examples_global)d new examples (buffer %(buffer)d), self-play %(self_play_s).2fs, "
                        "gather %(gather_s).3fs, train %(train_s).2fs (%(learner_steps)d steps), arena %(arena_s).2fs, "
                        "broadcast %(broadcast_s).3fs, win ratio %(win_ratio).2f, promoted %(promoted)s" % out)
        return out

    def run(self):
        for it in range(self.num_iterations):
            self.run_iteration(it)
        return self.history
