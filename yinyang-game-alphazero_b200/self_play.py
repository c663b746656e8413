"""Host-side mirror of src/yin_yang/ai/self_play.py: ``SelfPlayWorker`` / ``SelfPlayManager`` /
``generate_self_play_data`` with the reference's signatures and output format, driven by the batched engine
(``yy_selfplay_run``): all games of a call run concurrently on the GPU, one warp per game tree, leaves of all
games evaluated in one inference batch per simulation step.

Output (self_play.py:373-384): ``np.savez(boards=<object array of boards exposing .board / get_board()>,
policies=float64[N, A], values=float64[N])`` in ``<output_dir>/self_play_data_<unix time>.npz``.

Reference semantics kept (SURVEY section 3.5): search runs as player 1 for every ply while the move is applied
with the real player (Q5), every example of a game receives the same value (Q6), temperature 1 for the first
``temperature_threshold`` plies then argmax with random tie-break, Dirichlet noise only at ply 0.  Not kept:
the board-aliasing bug (Q1) -- stored boards are true snapshots of the position before each move.
"""
from __future__ import annotations

import logging
import os
import time

import numpy as np

from . import bitboard
from . import engine as _engine
from .game import YinYangLogic
from .network import YinYangNeuralNetwork

logger = logging.getLogger("YinYangSelfPlay")
MAX_CONCURRENT_GAMES = 4096          # game slots per GPU: 28 games per SM keep the tensor pipe of a B200 busy


def _load_network(game, model_path):
    """self_play.py:54-59; the width / depth of the network are taken from the checkpoint (the reference builds its
    default 128 x 10 network and fails on anything else)."""
    if os.path.exists(model_path):
        from . import weights as _weights
        from .network import safe_load
        sd = safe_load(model_path)["state_dict"]
        net = YinYangNeuralNetwork(game, *_weights.infer_arch(sd))
        net.load_state_dict(sd)
        logger.info(f"Loaded model from {model_path}")
    else:
        net = YinYangNeuralNetwork(game)
        logger.warning(f"No model found at {model_path}, using randomly initialized model")  # self_play.py:58-59
    return net


class RollingSelfPlay:
    """The game slots of one GPU, kept busy across calls (yy_selfplay_advance): every slot plays game after game at its
    own pace inside the persistent kernel; the host only launches, and drains the replay ring.

    ``advance(iterations)`` enqueues evaluation steps; ``drain()`` copies the records appended since the last drain to
    the host and returns the examples of every game that has FINISHED since (arrays, no per-example Python objects);
    ``play(num_games)`` runs until that many more games are complete.  With ``keep_warm=True`` the other slots keep
    their games in flight for the next call (a rolling generation has no tail); otherwise exactly ``num_games`` games
    are started (game quota) and the slots idle when they are done.

    ``full_search_prob`` < 1 turns on playout cap randomisation (Engine.selfplay_set_playout_cap): only that share of
    the moves gets the full ``num_simulations`` search and a record; the others get a fast search of
    ``fast_simulations`` (None: num_simulations) that only advances the game."""

    def __init__(self, game, state_dict=None, slots=MAX_CONCURRENT_GAMES, num_simulations=800, temperature_threshold=10,
                 dirichlet_alpha=0.3, dirichlet_epsilon=0.25, cpuct=1.0, seed=None, evaluator="nn", search_as_black=True,
                 device=None, replay_capacity=None, eval_symmetry="none", full_search_prob=1.0, fast_simulations=None):
        self.game = game
        self.n, self.m = game.getBoardSize()
        self.A = self.n * self.m
        self.slots, self.num_simulations = int(slots), int(num_simulations)
        if seed is None:
            seed = int(time.time_ns() & 0xFFFFFFFF)
        # a game makes at most ~2A moves (a move the real player cannot make is dropped but still searched: SURVEY Q5)
        self.max_moves = 2 * self.A + 4
        if replay_capacity is None:
            replay_capacity = self.slots * self.max_moves + 4096
        self.eng = _engine.Engine(rows=self.n, cols=self.m, n_games=self.slots, n_sims=self.num_simulations, evaluator=evaluator,
                                  cpuct=cpuct, rule_flags=getattr(game, "rule_flags", 0), search_as_black=search_as_black,
                                  dirichlet_alpha=dirichlet_alpha, dirichlet_epsilon=dirichlet_epsilon,
                                  temperature_threshold=temperature_threshold, seed=seed, state_dict=state_dict,
                                  replay_capacity=replay_capacity, device=device, eval_symmetry=eval_symmetry)
        if full_search_prob != 1.0 or fast_simulations is not None:
            self.eng.selfplay_set_playout_cap(full_search_prob, fast_simulations)
        self.cursor = 0                     # records drained so far
        self.games_requested = 0            # quota handed to the engine so far (exact mode)
        self.games_returned = 0
        self._pend = None                   # records of games still in progress
        self._stats = None

    def close(self):
        self.eng.close()

    def set_weights(self, state_dict):
        """New network for the games in flight and all later ones (H2D of the packed image)."""
        self.eng.load_state_dict(state_dict)

    def advance(self, iterations=None):
        self.eng.selfplay_advance(self.num_simulations + 1 if iterations is None else iterations)

    def drain(self):
        """-> dict(boards int8[E,n,m], pi float64[E,A], z float64[E], game int32[E], ply int16[E], player int8[E],
        counts uint16[E,A]) of the games finished since the last call, sorted by (game, ply); E may be 0.  With the
        playout cap on, a finished game may have no record at all: finished games are counted by the engine."""
        eng = self.eng
        st = self._stats = eng.stats()
        if st.examples - self.cursor > eng.replay_capacity:
            raise _engine._lib.YinYangError("replay ring overrun: drain more often or raise replay_capacity")
        new = eng.replay_window(self.cursor, st.examples)
        self.cursor = st.examples
        if self._pend is not None:
            new = {k: np.concatenate([self._pend[k], new[k]]) for k in new}
        results = _engine._to_host(eng.replay_views()["results"])[0]
        code = results[new["game_serial"] % eng.results_capacity] if len(new["ply"]) else np.zeros(0, np.int8)
        done = code != 0
        self._pend = {k: v[~done] for k, v in new.items()}
        idx = np.flatnonzero(done)
        idx = idx[np.lexsort((new["ply"][idx], new["game_serial"][idx]))]
        counts = new["counts"][idx]
        tot = counts.sum(axis=1, keepdims=True).astype(np.float64)
        pi = np.where(tot > 0, counts.astype(np.float64) / np.maximum(tot, 1), 1.0 / self.A)      # mcts.py:209-213
        out = {"boards": bitboard.unpack_boards(new["black"][idx], new["white"][idx], self.n, self.m), "pi": pi,
               "z": _engine.result_from_code(code[idx]), "game": new["game_serial"][idx], "ply": new["ply"][idx],
               "player": new["player"][idx], "counts": counts}
        self.games_returned = st.games_finished
        return out

    def play(self, num_games, keep_warm=False, poll_iterations=None):
        """Plays until ``num_games`` more games are complete and returns their examples (see drain)."""
        target = self.games_returned + num_games
        if keep_warm:
            self.eng.selfplay_set_quota(None)
        else:
            self.games_requested += num_games
            self.eng.selfplay_set_quota(self.games_requested)
        parts = []
        budget = (self.max_moves * (num_games // self.slots + 2)) * 2 * (self.num_simulations + 1)
        done_iters, step = 0, poll_iterations or max(self.num_simulations + 1, 256)
        while self.games_returned < target and done_iters < budget:
            self.advance(step)
            done_iters += step
            parts.append(self.drain())
            if self._stats.overflow:
                raise _engine._lib.YinYangError("a tree arena overflowed: raise edges_per_game")
        keys = parts[0].keys() if parts else ()
        return {k: np.concatenate([p[k] for p in parts]) for k in keys}


def play_games_arrays(game, state_dict, num_games, num_simulations=800, temperature_threshold=10, dirichlet_alpha=0.3,
                      dirichlet_epsilon=0.25, cpuct=1.0, seed=None, evaluator="nn", search_as_black=True, device=None,
                      max_slots=MAX_CONCURRENT_GAMES, eval_symmetry="none", full_search_prob=1.0, fast_simulations=None):
    """``num_games`` complete self-play games, all concurrent on the GPU; examples as arrays (RollingSelfPlay.drain).
    ``full_search_prob`` / ``fast_simulations``: playout cap randomisation (RollingSelfPlay)."""
    sp = RollingSelfPlay(game, state_dict, slots=max(1, min(num_games, max_slots)), num_simulations=num_simulations,
                         temperature_threshold=temperature_threshold, dirichlet_alpha=dirichlet_alpha,
                         dirichlet_epsilon=dirichlet_epsilon, cpuct=cpuct, seed=seed, evaluator=evaluator,
                         search_as_black=search_as_black, device=device, eval_symmetry=eval_symmetry,
                         full_search_prob=full_search_prob, fast_simulations=fast_simulations)
    try:
        return sp.play(num_games)
    finally:
        sp.close()


def play_games(game, state_dict, num_games, num_simulations=800, temperature_threshold=10, dirichlet_alpha=0.3,
               dirichlet_epsilon=0.25, cpuct=1.0, seed=None, evaluator="nn", search_as_black=True, max_moves=None,
               device=None, full_search_prob=1.0, fast_simulations=None):
    """Plays ``num_games`` complete self-play games concurrently.  Returns a list (one entry per game, in game
    order) of example lists ``[(YinYangLogic, pi float64[A], z float), ...]`` -- the reference's per-game return value
    (self_play.py:72-192); ``play_games_arrays`` is the same without the per-example objects.  With the playout cap on
    (``full_search_prob`` < 1) a game's list holds its full-search moves only, and may be empty."""
    n, m = game.getBoardSize()
    ex = play_games_arrays(game, state_dict, num_games, num_simulations, temperature_threshold, dirichlet_alpha,
                           dirichlet_epsilon, cpuct, seed, evaluator, search_as_black, device,
                           full_search_prob=full_search_prob, fast_simulations=fast_simulations)
    games = [[] for _ in range(num_games)]
    rule_flags = getattr(game, "rule_flags", 0)
    for i in range(len(ex["z"])):
        b = YinYangLogic(n, m, rule_flags)
        b.board = ex["boards"][i].copy()
        z = float(ex["z"][i])
        games[int(ex["game"][i])].append((b, ex["pi"][i].copy(), z if z == 0.0001 else int(z)))
    return games


class SelfPlayWorker:
    """self_play.py:22-216.  ``play_game`` plays one game; ``generate_games`` plays ``num_games`` concurrently."""

    def __init__(self, game, model_path, num_simulations=800, num_games=1, temperature_threshold=10,
                 dirichlet_alpha=0.3, dirichlet_epsilon=0.25, cpuct=1.0, num_parallel=1):
        self.game, self.model_path = game, model_path
        self.num_simulations, self.num_games = num_simulations, num_games
        self.temperature_threshold = temperature_threshold
        self.dirichlet_alpha, self.dirichlet_epsilon, self.cpuct = dirichlet_alpha, dirichlet_epsilon, cpuct
        self.num_parallel = num_parallel
        self.neural_net = _load_network(game, model_path)

    def _play(self, count):
        return play_games(self.game, self.neural_net.state_dict(), count, self.num_simulations, self.temperature_threshold,
                          self.dirichlet_alpha, self.dirichlet_epsilon, self.cpuct)

    def play_game(self):
        return self._play(1)[0]

    def generate_games(self):
        all_examples = []
        for i, ex in enumerate(self._play(self.num_games)):
            all_examples.extend(ex)
            logger.info(f"Completed game {i + 1}/{self.num_games} with {len(ex)} examples")
        return all_examples


class SelfPlayManager:
    """self_play.py:218-335.  ``num_workers`` x ``games_per_worker`` games; the reference forks one process per
    worker -- here they all share the GPU batch (the worker count only determines how many games are played)."""

    def __init__(self, game, model_path, num_workers=1, num_simulations=800, games_per_worker=1,
                 temperature_threshold=10, dirichlet_alpha=0.3, dirichlet_epsilon=0.25, cpuct=1.0, mcts_parallel=1):
        self.game, self.model_path = game, model_path
        self.num_workers, self.num_simulations, self.games_per_worker = num_workers, num_simulations, games_per_worker
        self.temperature_threshold = temperature_threshold
        self.dirichlet_alpha, self.dirichlet_epsilon, self.cpuct = dirichlet_alpha, dirichlet_epsilon, cpuct
        self.mcts_parallel = mcts_parallel

    def generate_games_parallel(self):
        try:
            worker = SelfPlayWorker(self.game, self.model_path, self.num_simulations, self.num_workers * self.games_per_worker,
                                    self.temperature_threshold, self.dirichlet_alpha, self.dirichlet_epsilon, self.cpuct)
            examples = worker.generate_games()
        except Exception as e:  # self_play.py:283-286: a failed worker contributes no examples
            logger.error(f"Self-play failed: {e}")
            examples = []
        logger.info(f"Generated {len(examples)} examples")
        return examples


def save_examples(filename, examples, action_size, wire="native"):
    """np.savez(boards=<object array>, policies=float64[N,A], values=float64[N]) (self_play.py:373-384).

    wire="native"    : boards are this package's ``YinYangLogic`` (unpickling needs ``yy_b200`` importable);
    wire="reference" : boards are pickled as ``src.yin_yang.yin_yang_logic.YinYangLogic`` (attributes n, m, board:
                       yin_yang_logic.py:14-22), so the reference's own trainer (``TrainingDataQueue.push_file``,
                       training_pipeline.py:55-73) loads the file without this package installed."""
    boards = np.empty(len(examples), dtype=object)
    undo = None
    if wire == "reference":
        cls, undo = _reference_board_class()
        for i, ex in enumerate(examples):
            o = cls.__new__(cls)
            o.n, o.m = int(ex[0].n), int(ex[0].m)
            o.board = np.array(ex[0].get_board() if hasattr(ex[0], "get_board") else ex[0].board, dtype=np.int8)
            boards[i] = o
    elif wire == "native":
        for i, ex in enumerate(examples):
            boards[i] = ex[0]
    else:
        raise ValueError("wire must be 'native' or 'reference'")
    policies = np.array([ex[1] for ex in examples], dtype=np.float64).reshape(len(examples), action_size)
    values = np.array([ex[2] for ex in examples], dtype=np.float64)
    try:
        np.savez(filename, boards=boards, policies=policies, values=values)
    finally:
        if undo:
            import sys
            for name in undo:
                sys.modules.pop(name, None)
    return filename


def _reference_board_class():
    """(class, fake module names to remove afterwards).  pickle stores a class by module path + name and checks that the
    path resolves to the very object being pickled: use the reference's class when it is importable, otherwise register
    a stand-in under the reference's module path for the duration of the save."""
    import sys
    import types
    try:
        from src.yin_yang.yin_yang_logic import YinYangLogic as Ref   # running inside the reference tree
        return Ref, None
    except Exception:
        created = []
        for name in ("src", "src.yin_yang", "src.yin_yang.yin_yang_logic"):
            if name not in sys.modules:
                sys.modules[name] = types.ModuleType(name)
                created.append(name)
        cls = type("YinYangLogic", (), {"__module__": "src.yin_yang.yin_yang_logic"})
        sys.modules["src.yin_yang.yin_yang_logic"].YinYangLogic = cls
        return cls, created


def save_example_arrays(filename, ex, n, m, wire="arrays", rule_flags=0):
    """The same file from example ARRAYS (RollingSelfPlay.drain / play_games_arrays).  wire="arrays" stores the boards as
    one int8[N, n, m] array under the reference's key -- no per-example objects at all; this package's
    TrainingDataQueue.push_file reads it; "native" / "reference" build the object array the reference's format wants."""
    if wire == "arrays":
        np.savez(filename, boards=np.ascontiguousarray(ex["boards"], dtype=np.int8), policies=np.asarray(ex["pi"], dtype=np.float64),
                 values=np.asarray(ex["z"], dtype=np.float64))
        return filename
    examples = []
    for i in range(len(ex["z"])):
        b = YinYangLogic(n, m, rule_flags)
        b.board = ex["boards"][i].copy()
        examples.append((b, ex["pi"][i], ex["z"][i]))
    return save_examples(filename, examples, n * m, wire)


def generate_self_play_data(game, model_path, output_dir, num_games=100, num_workers=1, num_simulations=800, wire="native", file_tag="",
                            eval_symmetry="none", full_search_prob=1.0, fast_simulations=None):
    """self_play.py:337-387.  Returns the path of the written .npz (``wire``: see save_examples / save_example_arrays;
    ``file_tag``: suffix that keeps the files of several ranks apart).  num_workers x (num_games // num_workers) games
    (self_play.py:355), all concurrent on the GPU.  ``full_search_prob`` / ``fast_simulations``: playout cap randomisation
    (RollingSelfPlay)."""
    os.makedirs(output_dir, exist_ok=True)
    games_per_worker = max(1, num_games // num_workers)          # self_play.py:355
    n, m = game.getBoardSize()
    try:
        net = _load_network(game, model_path)
        ex = play_games_arrays(game, net.state_dict(), num_workers * games_per_worker, num_simulations, eval_symmetry=eval_symmetry,
                               full_search_prob=full_search_prob, fast_simulations=fast_simulations)
    except Exception as e:  # self_play.py:283-286: a failed worker contributes no examples
        logger.error(f"Self-play failed: {e}")
        ex = {"boards": np.zeros((0, n, m), np.int8), "pi": np.zeros((0, n * m)), "z": np.zeros(0)}
    filename = os.path.join(output_dir, f"self_play_data_{int(time.time())}{file_tag}.npz")
    save_example_arrays(filename, ex, n, m, wire, getattr(game, "rule_flags", 0))
    logger.info(f"Saved {len(ex['z'])} examples to {filename}")
    return filename


def generate_self_play_data_distributed(game, model_path, output_dir, num_games=100, num_simulations=800, wire="arrays",
                                        backend=None, eval_symmetry="none", full_search_prob=1.0, fast_simulations=None):
    """generate_self_play_data for one process per GPU (``torchrun``): every rank plays its contiguous share of the
    ``num_games`` games with its own random streams, the examples are gathered to rank 0 (NCCL all-gather of the record
    tensors; gloo in the CPU tests' plumbing check) and rank 0 writes ONE ``self_play_data_<time>.npz``.  Initialises the
    process group from the torchrun environment when there is none.  Returns the file path on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist
    from . import distributed as yyd
    own_group = not dist.is_initialized()
    if own_group:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group(backend or "nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    n, m = game.getBoardSize()
    lo, hi = yyd.shard_games(num_games, world, rank)
    net = _load_network(game, model_path)
    t = torch.tensor([time.time_ns() & 0xFFFFFFFF], dtype=torch.int64, device="cuda")
    dist.broadcast(t, 0)                                              # one base seed for the job, a distinct stream per rank
    seed = yyd.rank_seed(int(t.item()), rank) & 0x7FFFFFFFFFFFFFFF
    if hi > lo:
        ex = play_games_arrays(game, net.state_dict(), hi - lo, num_simulations, seed=seed, eval_symmetry=eval_symmetry,
                               full_search_prob=full_search_prob, fast_simulations=fast_simulations)
    else:
        ex = {"boards": np.zeros((0, n, m), np.int8), "pi": np.zeros((0, n * m)), "z": np.zeros(0), "game": np.zeros(0, np.int32),
              "counts": np.zeros((0, n * m), np.uint16)}
    dev = torch.device("cuda")
    rec = {"boards": torch.from_numpy(np.ascontiguousarray(ex["boards"], dtype=np.int8)).to(dev),
           "counts": torch.from_numpy(np.ascontiguousarray(ex["counts"]).view(np.int16)).to(dev),
           "z": torch.from_numpy(np.asarray(ex["z"], dtype=np.float64)).to(dev),
           "game": torch.from_numpy(np.asarray(ex["game"], dtype=np.int32) + lo).to(dev)}
    out = yyd.gather_records(rec, dst=0)
    path = None
    if rank == 0:
        counts = out["counts"].cpu().numpy().view(np.uint16)
        tot = counts.sum(axis=1, keepdims=True).astype(np.float64)
        allx = {"boards": out["boards"].cpu().numpy(), "z": out["z"].cpu().numpy(),
                "pi": np.where(tot > 0, counts.astype(np.float64) / np.maximum(tot, 1), 1.0 / (n * m))}
        os.makedirs(output_dir, exist_ok=True)
        path = os.path.join(output_dir, f"self_play_data_{int(time.time())}.npz")
        save_example_arrays(path, allx, n, m, wire, getattr(game, "rule_flags", 0))
        logger.info(f"Saved {len(allx['z'])} examples of {num_games} games from {world} ranks to {path}")
    dist.barrier()
    if own_group:
        dist.destroy_process_group()
    return path
