"""The board-form map and the random-form hash of the product header (yy_rules.cuh), compiled for the host, against
numpy's rot90 / flip / transpose forms, the oracle's augmentation and a Python restatement of the hash (no GPU)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import symmetry_ref as S
from conftest import ROOT, random_play_boards

SUPPORTED = [(n, m) for n in range(1, 33) for m in range(1, 33) if n * m <= 256]


@pytest.fixture(scope="module")
def forms_lib():
    d = os.path.join(ROOT, "tests", "_host")
    so = os.path.join(d, "libforms_host.so")
    src = os.path.join(d, "forms_host_shim.cpp")
    hdr = os.path.join(ROOT, "yinyang-game-alphazero_b200", "csrc", "yy_rules.cuh")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def _form_src(lib, f, n, m):
    out = np.zeros(n * m, dtype=np.int32)
    rc = lib.yyh_form_src(f, n, m, out.ctypes.data_as(ctypes.c_void_p))
    return out if rc == 0 else None


def test_form_map_matches_numpy_forms(forms_lib):
    """Every supported board and form: the header's map is numpy's form of the cell-index grid; forms that change a
    rectangular board's shape are refused."""
    for n, m in SUPPORTED:
        for f in range(8):
            got = _form_src(forms_lib, f, n, m)
            if f not in S.forms(n, m):
                assert got is None, (n, m, f)
                continue
            ref = S.transform(np.arange(n * m).reshape(n, m), f)
            assert ref.shape == (n, m), (n, m, f)
            assert np.array_equal(got, ref.reshape(-1)), (n, m, f)
            assert np.array_equal(np.sort(got), np.arange(n * m)), (n, m, f)


@pytest.mark.parametrize("n", [4, 6, 8, 16])
def test_form_map_is_the_augmentation_permutation(forms_lib, oracle_mod, n):
    """The oracle's augment_dataset (the restatement the golden augmentation tests hold yy_augment_samples to) writes
    form f's planes and policy as the record's, permuted by the header's map."""
    boards, _ = random_play_boards(oracle_mod, n, n, 6, seed=n)
    counts = np.random.default_rng(n).integers(0, 50, size=(6, n * n))
    planes, pol, _ = oracle_mod.augment_dataset(boards, counts, np.zeros(6), n, n)
    planes = planes.reshape(6, 8, 5, n * n)
    pol = pol.reshape(6, 8, n * n)
    for f in range(8):
        src = _form_src(forms_lib, f, n, n)
        assert np.array_equal(planes[:, f], planes[:, 0][..., src]), f
        assert np.array_equal(pol[:, f], pol[:, 0][..., src]), f


@pytest.mark.parametrize("n,m", [(8, 8), (6, 6), (16, 16), (5, 7), (10, 8), (1, 1), (3, 22), (12, 12)])
def test_form_hash_matches_restatement(forms_lib, oracle_mod, yy, n, m):
    """forms[mix64(stub_key(board) ^ seed) % F]: the host-compiled C function against the oracle's stub key and a Python
    mix64 on random positions and seeds (including the top bit of the seed)."""
    boards, _ = random_play_boards(oracle_mod, n, m, 64, seed=n * 31 + m)
    b, w = yy.bitboard.pack_boards(boards, n, m)
    for seed in (0, 1, 12345, 0xFEDCBA9876543210):
        out = np.zeros(len(boards), dtype=np.int32)
        assert forms_lib.yyh_hashed_form(n, m, b.ctypes.data_as(ctypes.c_void_p), w.ctypes.data_as(ctypes.c_void_p),
                                         ctypes.c_long(len(boards)), ctypes.c_uint64(seed), out.ctypes.data_as(ctypes.c_void_p)) == 0
        ref = [S.hashed_form(bd, n, m, seed) for bd in boards]
        assert out.tolist() == ref, seed
    if n * m >= 16:
        assert len(set(out.tolist())) > 1, "the hash should spread positions over the forms"
