"""Host-side mirror of src/yin_yang/ai/mcts.py: same constructor keywords, ``search`` / ``select_action`` /
``reuse_tree`` and a ``root`` object with the statistics the reference's callers read -- the search itself
(select / expand / backup, HBM-resident tree) runs in ``libyinyang_b200.so``.

Evaluator seam (duck typing, like the reference: anything with ``predict(board) -> (policy[A], value)``):
  * ``network.YinYangNeuralNetwork``  -> fused on-device bf16 inference (evaluator "nn");
  * ``network.HashStubEvaluator``     -> on-device deterministic priors (evaluator "stub", bit-exact parity mode);
  * any other object with ``predict`` -> "external": the tree stays on the GPU, each pending leaf is handed to
    ``predict`` on the host and its priors/value are uploaded (yy_search_begin / yy_search_advance).
The Game must be a ``game.YinYangGame`` (the rules run on the GPU); arbitrary Python games are out of scope.
"""
from __future__ import annotations

import logging

import numpy as np
import torch

from . import bitboard, engine as _engine
from .network import HashStubEvaluator, YinYangNeuralNetwork

logger = logging.getLogger("YinYangMCTS")
CPUCT = 1.0  # mcts.py:26


class Node:
    """Read-only mirror of the reference's Node (mcts.py:28-225) over the engine's tree arrays (Engine.tree_host): the
    statistics its callers and tests read -- ``visits``, ``value_sum`` (np.float32, SURVEY Q4), ``prior``, ``children``
    (dict action -> Node in ascending action order, built on first access, the whole tree is reachable), ``board``,
    ``player``, ``is_terminal`` / ``terminal_value``, ``is_expanded()``, ``get_children_visit_counts()``,
    ``get_children_distribution(temperature)``."""

    def __init__(self, game, tree, node_id, visits, value_sum=0.0, prior=0.0, action=None, parent=None):
        self.game, self._t, self._id = game, tree, int(node_id)
        self.visits, self.value_sum, self.prior = int(visits), np.float32(value_sum), np.float32(prior)
        self.action, self.parent = action, parent
        self._children = None

    # -- state of the node (None / False while no simulation has expanded it: mcts.py:42-48)
    @property
    def player(self):
        return int(self._t["player"][self._id]) if self._id >= 0 else None

    @property
    def board(self):
        if self._id < 0:
            return None
        from .game import YinYangLogic
        n, m = self.game.getBoardSize()
        b = YinYangLogic(n, m, getattr(self.game, "rule_flags", 0))
        b.board = bitboard.unpack_boards(self._t["black"][self._id][None], self._t["white"][self._id][None], n, m)[0]
        return b

    @property
    def is_terminal(self):
        return self._id >= 0 and bool(self._t["flags"][self._id] & 2)

    @property
    def terminal_value(self):
        if not self.is_terminal:
            return None
        v = float(self._t["value"][self._id])
        return int(v) if v in (1.0, -1.0) else 0.0001          # yin_yang_game.py:101-107

    @property
    def children(self):
        if self._children is None:
            self._children = {}
            if self._id >= 0:
                t, base, cnt = self._t, int(self._t["edge_base"][self._id]), int(self._t["n_edges"][self._id])
                for k in range(base, base + cnt):
                    a = int(t["action"][k])
                    self._children[a] = Node(self.game, t, t["child"][k], t["N"][k], t["W"][k], t["P"][k], a, self)
        return self._children

    def is_expanded(self):  # mcts.py:93-95
        return len(self.children) > 0

    def get_value(self):  # mcts.py:158-162
        return 0.0 if self.visits == 0 else self.value_sum / self.visits

    def get_visit_count(self):
        return self.visits

    def get_children_visit_counts(self):  # mcts.py:168-181
        counts = np.zeros(self.game.getActionSize())
        for a, ch in self.children.items():
            counts[a] = ch.visits
        return counts

    def get_children_distribution(self, temperature=1.0):  # mcts.py:183-215
        counts = self.get_children_visit_counts()
        A = counts.size
        if temperature == 0:
            best = np.where(counts == np.max(counts))[0]
            probs = np.zeros(A)
            probs[best] = 1.0 / len(best)
            return probs
        if temperature != 1.0:
            counts = np.power(counts, 1.0 / temperature)
        s = np.sum(counts)
        return counts / s if s > 0 else np.ones(A) / A


ChildStats = RootView = Node      # names of the round-1 facade


class MCTS:
    def __init__(self, game, neural_net, num_simulations=800, cpuct=1.0, temperature=1.0, num_threads=1,
                 dirichlet_noise=True, dirichlet_alpha=0.3, dirichlet_epsilon=0.25, verbose=1, eval_symmetry="none"):
        self.game, self.neural_net = game, neural_net
        # network evaluations of the leaves: "none" as they are, "random" in one dihedral form hashed from (seed, position),
        # "average" averaged over all forms (Engine(eval_symmetry=); network evaluator only)
        self.eval_symmetry = eval_symmetry
        self.num_simulations, self.cpuct, self.temperature = num_simulations, cpuct, temperature
        # mcts.py:320-321,414-426 runs the simulations of a search on `num_threads` threads; here num_threads = K > 1 selects
        # K leaves per game per step with virtual loss (Engine(leaves_per_step=K)): K simulations share one network batch,
        # which cuts the latency of a single-position search; 1 (default) = the exact sequential search
        self.num_threads = max(1, num_threads)
        self.use_dirichlet, self.dirichlet_alpha, self.dirichlet_epsilon = dirichlet_noise, dirichlet_alpha, dirichlet_epsilon
        self._engines = {}
        logger.setLevel({0: logging.ERROR, 1: logging.INFO}.get(verbose, logging.DEBUG))

    # -- engine per batch size
    def _mode(self):
        if isinstance(self.neural_net, YinYangNeuralNetwork):
            return "nn"
        if isinstance(self.neural_net, HashStubEvaluator):
            return "stub"
        return "external"

    def _engine(self, n_games):
        e = self._engines.get(n_games)
        version = getattr(self.neural_net, "weights_version", 0)
        if e is not None and self._mode() == "nn" and getattr(e, "_weights_version", version) != version:
            e.load_state_dict(self.neural_net.state_dict())      # the net was reloaded / trained since the engine was built:
            e._weights_version = version                         # the reference holds the net by reference (mcts.py:249)
        if e is None:
            n, m = self.game.getBoardSize()
            kw = dict(rows=n, cols=m, n_games=n_games, n_sims=self.num_simulations, evaluator=self._mode(), cpuct=self.cpuct,
                      rule_flags=getattr(self.game, "rule_flags", 0), dirichlet_alpha=self.dirichlet_alpha,
                      dirichlet_epsilon=self.dirichlet_epsilon)
            if self._mode() == "nn":
                kw["state_dict"] = self.neural_net.state_dict()
            if self.eval_symmetry != "none":
                kw["eval_symmetry"] = self.eval_symmetry
            if self.num_threads > 1 and self._mode() != "external":
                kw["leaves_per_step"] = self.num_threads
            e = self._engines[n_games] = _engine.Engine(**kw)
            e._weights_version = version
        return e

    # -- batched search: the natural GPU entry point
    def search_batch(self, grids, players, add_exploration_noise=False):
        """grids int8[B,n,m], players [B] -> (counts int32[B,A], child value sums float32[B,A])."""
        grids = np.asarray(grids, np.int8)
        players = np.asarray(players, np.int8)
        B = grids.shape[0]
        e = self._engine(B)
        n, m = self.game.getBoardSize()
        noise = None
        if add_exploration_noise and self.use_dirichlet:  # mcts.py:298-312: np.random.dirichlet over the legal actions
            masks = _engine.legal_mask_host(grids, players, n, m, getattr(self.game, "rule_flags", 0))
            noise = [np.random.dirichlet([self.dirichlet_alpha] * int(mk.sum())) if mk.any() else None for mk in masks]
        if self._mode() != "external":
            return e.search_host(grids, players, noise=noise)
        return self._search_external(e, grids, players, noise)

    def _search_external(self, e, grids, players, noise):
        n, m = self.game.getBoardSize()
        A, B = n * m, grids.shape[0]
        b, w = bitboard.pack_boards(grids, n, m)
        bd, wd = torch.from_numpy(b.view(np.int64)).cuda(), torch.from_numpy(w.view(np.int64)).cuda()
        nz = nm = None
        if noise is not None:
            full, mask = np.zeros((B, A)), np.zeros(B, np.uint8)
            for g, v in enumerate(noise):
                if v is not None:
                    full[g, : len(v)], mask[g] = v, 1
            nz, nm = torch.from_numpy(full).cuda(), torch.from_numpy(mask).cuda()
        e.search_begin(bd, wd, torch.from_numpy(players).cuda(), nz, nm)
        active = B
        from .game import YinYangLogic
        while active:
            lb, lw, act = e.leaf_batch()
            leaf = bitboard.unpack_boards(lb.cpu().numpy().view(np.uint64), lw.cpu().numpy().view(np.uint64), n, m)
            pending = act.cpu().numpy()
            pri, val = np.zeros((B, A), np.float32), np.zeros(B, np.float32)
            for g in np.flatnonzero(pending):
                board = YinYangLogic(n, m)
                board.board = leaf[g]
                p, v = self.neural_net.predict(board)   # the duck-typed seam (mcts.py:295,394)
                pri[g], val[g] = np.asarray(p, np.float32), np.float32(v)
            active = e.search_advance(torch.from_numpy(pri).cuda(), torch.from_numpy(val).cuda())
        counts, cw = e.search_counts()
        return counts.cpu().numpy(), cw.cpu().numpy()

    # -- reference surface
    def search(self, board, player, add_exploration_noise=False):  # mcts.py:275-343
        n, m = self.game.getBoardSize()
        grid = board.get_board()
        counts, cw = self.search_batch(grid[None], [player], add_exploration_noise)
        # the tree stays in the engine's arenas until the next search: mirror it (root.visits = simulations run, mcts.py:406-412)
        root = Node(self.game, self._engine(1).tree_host(0), 0, self.num_simulations)
        logger.info("MCTS search completed with %d total visits", root.visits)
        return root.get_children_distribution(self.temperature), root

    def select_action(self, board, player, temperature=None, valid_moves=None, add_exploration_noise=False):  # mcts.py:427-479
        temp = temperature if temperature is not None else self.temperature
        action_probs, _ = self.search(board, player, add_exploration_noise)
        if valid_moves is not None:
            if len(valid_moves) != len(action_probs):
                valid_moves = np.ones_like(action_probs)
            masked = action_probs * valid_moves
            s = np.sum(masked)
            if s <= 0:
                return int(np.argmax(action_probs))
            action_probs = masked / s
        if temp == 0:
            return int(np.argmax(action_probs))
        return int(np.random.choice(np.arange(len(action_probs)), p=action_probs))

    def reuse_tree(self, old_root, board, player, action_taken):  # mcts.py:481-505
        """The reference never feeds the returned node back into ``search`` (self_play.py:134-137,192; SURVEY Q7),
        so reuse is a no-op there too; kept for interface parity."""
        if old_root is not None and action_taken in getattr(old_root, "children", {}):
            child = old_root.children[action_taken]
            child.parent = None
            return child
        return None

    def close(self):
        for e in self._engines.values():
            e.close()
        self._engines.clear()
