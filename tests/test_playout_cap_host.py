"""The playout-cap decision full(s, p) (DESIGN.md §3.3): its Python restatement at the ends of the range and its
frequency, and the product header's function (yy_rules.cuh: playout_full), compiled for the host, against it (no GPU)."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

import playout_cap_ref as P
from conftest import ROOT

SEEDS = (0, 7, 12345, 0xFEDCBA9876543210)


@pytest.fixture(scope="module")
def cap_lib():
    d = os.path.join(ROOT, "tests", "_host")
    so = os.path.join(d, "libplayout_cap_host.so")
    src = os.path.join(d, "playout_cap_host_shim.cpp")
    hdr = os.path.join(ROOT, "yinyang-game-alphazero_b200", "csrc", "yy_rules.cuh")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def _pairs(count, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 1 << 20, size=count).astype(np.int32), rng.integers(0, 600, size=count).astype(np.int32)


def test_threshold_is_llround():
    assert P.threshold(1.0) == 1 << 32 and P.threshold(0.0) == 0 and P.threshold(0.25) == 1 << 30
    assert P.threshold(0.5 / 2 ** 32) == 1 and P.threshold(0.49 / 2 ** 32) == 0


def test_always_full_at_one_and_never_at_zero():
    serials, plies = _pairs(2000, 1)
    for seed in SEEDS:
        assert all(P.full(seed, int(s), int(p), 1.0) for s, p in zip(serials, plies))
        assert not any(P.full(seed, int(s), int(p), 0.0) for s, p in zip(serials, plies))


@pytest.mark.parametrize("p_full", [0.25, 0.5])
def test_full_fraction_is_binomial(p_full):
    """Over 100,000 (serial, ply) pairs -- every ply of 1,000 consecutive games -- the share of full searches lies within
    5 sigma of p_full."""
    n = 100_000
    hits = sum(P.full(99, s, p, p_full) for s in range(1000) for p in range(100))
    sigma = math.sqrt(n * p_full * (1 - p_full))
    assert abs(hits - n * p_full) < 5 * sigma, hits


@pytest.mark.parametrize("p_full", [0.0, 0.05, 0.25, 0.5, 0.999, 1.0])
def test_header_function_matches_restatement(cap_lib, p_full):
    serials, plies = _pairs(5000, int(p_full * 1000) + 3)
    serials[:4] = [0, 1, 0x7FFFFFFF, 4095]
    plies[:4] = [0, 0, 1, 0xFFFFF]
    T = P.threshold(p_full)
    for seed in SEEDS:
        out = np.zeros(len(serials), dtype=np.uint8)
        cap_lib.yyh_playout_full(ctypes.c_uint64(seed), serials.ctypes.data_as(ctypes.c_void_p), plies.ctypes.data_as(ctypes.c_void_p),
                                 ctypes.c_long(len(serials)), ctypes.c_uint64(T), out.ctypes.data_as(ctypes.c_void_p))
        ref = [P.full(seed, int(s), int(p), p_full) for s, p in zip(serials, plies)]
        assert out.astype(bool).tolist() == ref, seed


@pytest.mark.parametrize("n,m,sims,sab", [(4, 4, 30, True), (5, 5, 20, False)])
def test_reference_game_without_cap_is_the_oracle_game(oracle_mod, n, m, sims, sab):
    """The capped restatement with every ply full is oracle.play_game, move for move."""
    rng = np.random.default_rng(n * 10 + m)
    for s in range(3):
        uniforms, noise = rng.random(4 * n * m), rng.dirichlet([0.3] * (n * m))
        b, pi, z, kind = oracle_mod.play_game(n, m, sims, uniforms, noise, temperature_threshold=4, search_as_black=sab)
        rb, rpi, rz, rkind, full_plies, fast_plies, result = P.play_game(n, m, sims, uniforms, noise, temperature_threshold=4,
                                                                         search_as_black=sab)
        assert np.array_equal(b, rb) and np.array_equal(pi, rpi) and np.array_equal(z, rz) and kind == rkind
        assert full_plies == list(range(len(b))) and fast_plies == [] and np.all(z == result)


def test_reference_game_fast_plies_are_not_recorded(oracle_mod):
    """With every other ply fast, the recorded plies are the even ones and each is the oracle's full search there."""
    n = m = 4
    rng = np.random.default_rng(5)
    uniforms, noise = rng.random(64), rng.dirichlet([0.3] * 16)
    b, pi, z, kind, full_plies, fast_plies, result = P.play_game(n, m, 30, uniforms, noise, playout_cap=(3, lambda p: p % 2 == 0))
    assert full_plies == list(range(0, 2 * len(full_plies), 2)) and all(p % 2 == 1 for p in fast_plies)
    assert len(b) == len(full_plies) and np.all(z == result)
    r = oracle_mod.mcts_search(b[0], 1, n, m, 30, noise=noise)
    assert np.array_equal(pi[0], r["counts"] / r["counts"].sum())
