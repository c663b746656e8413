"""Reference restatement of playout cap randomisation (DESIGN.md §3.3): which self-play moves get the full search, and
the oracle's whole game (oracle.play_game) with fast searches that are played but not recorded."""
import math

import numpy as np

from symmetry_ref import MASK64, mix64

PLAYOUT_SALT = 0x706C61796F757463      # "playoutc"


def threshold(p_full):
    """T = llround(p_full * 2^32): the nearest integer, halves away from zero (p_full * 2^32 is exact in float64)."""
    x = float(p_full) * 2.0 ** 32
    f = math.floor(x)
    return int(f) + (1 if x - f >= 0.5 else 0)


def full(seed, serial, ply, p_full):
    """Is the move of game `serial` at ply `ply` a full search under engine seed `seed`?"""
    key = mix64(mix64((seed & MASK64) ^ PLAYOUT_SALT) ^ (((serial & 0xFFFFFFFF) << 20) | ply))
    return (key >> 32) < threshold(p_full)


def play_game(n, m, num_sims, uniforms, noise=None, cpuct=1.0, eps=0.25, temperature_threshold=10, rule_flags=0,
              search_as_black=True, playout_cap=None):
    """oracle.play_game with a playout cap: playout_cap = (fast_sims, full_fn), full_fn(step) -> bool.  A full step is the
    oracle's step; a fast step searches with fast_sims simulations and no noise and appends nothing to the examples --
    its action choice, apply and terminal test are the same.  None = every step full (oracle.play_game).
    Returns (boards, pis, zs, end, full_plies, fast_plies, result): the recorded examples as oracle.play_game returns
    them, the plies that were full / fast searches, and the game's result (the z of every example; also defined for a
    game without any)."""
    import oracle
    fast_sims, full_fn = playout_cap if playout_cap is not None else (num_sims, lambda step: True)
    A = n * m
    board = np.zeros((n, m), dtype=np.int8)
    player, step, passes = 1, 0, 0
    boards, pis, full_plies, fast_plies = [], [], [], []

    def finish(result, kind):
        zs, value = [], result
        for i in range(len(boards)):                      # self_play.py:112-115 / :172-181
            zs.append(value if i % 2 == 0 else -value)
            value = -value
        return (np.array(boards, dtype=np.int8).reshape(-1, n, m), np.array(pis, dtype=np.float64).reshape(-1, A),
                np.array(zs, dtype=np.float64), kind, full_plies, fast_plies, result)

    while True:
        temperature = 1.0 if step < temperature_threshold else 0
        sp = 1 if search_as_black else player
        valid = oracle.legal_mask(board[None], np.array([sp], np.int8), n, m, rule_flags)[0].astype(np.float64)
        idx = np.flatnonzero(valid == 1)
        if len(idx) == 0:
            passes += 1
            if passes >= 2:
                result = float(oracle.game_ended(board[None], np.array([player], np.int8), n, m, rule_flags)[0])
                if result == 0:
                    result = 1e-4
                return finish(result, "passes")
            player = -player
            continue
        passes = 0
        is_full = bool(full_fn(step))
        r = oracle.mcts_search(board, sp, n, m, num_sims if is_full else fast_sims, cpuct=cpuct, rule_flags=rule_flags,
                               noise=noise if (is_full and step == 0 and noise is not None) else None, eps=eps)
        counts = r["counts"].astype(np.float64)
        pi = counts / counts.sum() if counts.sum() > 0 else np.ones(A) / A      # mcts.py:207-213 (temperature 1)
        if is_full:
            boards.append(board.copy()); pis.append(pi); full_plies.append(step)
        else:
            fast_plies.append(step)
        u = float(uniforms[step])
        if temperature == 0:
            best = np.flatnonzero(pi == pi.max())
            action = int(best[oracle.choice_index(u, k=len(best))])
        else:
            probs = pi * valid
            if probs.sum() > 0:
                probs = probs / probs.sum()
            else:
                probs = np.zeros_like(valid); probs[idx] = 1.0 / len(idx)
            action = oracle.choice_index(u, p=probs)
        nb, npl = oracle.next_state(board[None], np.array([player], np.int8), np.array([action], np.int32), n, m, rule_flags)
        board, player = nb[0], int(npl[0])
        step += 1
        result = float(oracle.game_ended(board[None], np.array([player], np.int8), n, m, rule_flags)[0])
        if result != 0:
            return finish(result, "ended")
