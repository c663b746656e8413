"""Reference restatement of symmetric evaluation (DESIGN.md §3.2.1): the dihedral forms of a board in augment_sample's
order, the map from a form's cells back to the board's actions, and the random-form hash
forms[mix64(stub_key(board) ^ seed) % F] with the oracle's stub key."""
import ctypes

import numpy as np

MASK64 = (1 << 64) - 1


def forms(n, m):
    """Forms that keep an n x m board's shape: all 8 on square boards, {0, 2, 4, 5} otherwise."""
    return list(range(8)) if n == m else [0, 2, 4, 5]


def transform(g, f):
    """Form f of an array [..., n, m] (oracle._symmetries / augment_sample order)."""
    from oracle import _symmetries
    return np.ascontiguousarray(_symmetries(np.asarray(g))[f])


def src_map(n, m, f):
    """int64[A]: cell c of form f shows cell src[c] of the board (T_f(b).ravel() == b.ravel()[src])."""
    return transform(np.arange(n * m).reshape(n, m), f).reshape(-1)


def unmap(out_f, n, m, f):
    """Outputs of the network on T_f(b), indexed by the board's own actions: result[..., src[c]] = out_f[..., c]."""
    res = np.empty_like(out_f)
    res[..., src_map(n, m, f)] = out_f
    return res


def mix64(z):
    z = (z + 0x9E3779B97F4A7C15) & MASK64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK64
    return z ^ (z >> 31)


def stub_key(board, n, m):
    import oracle
    b = np.ascontiguousarray(board, dtype=np.int8).reshape(-1)
    return int(oracle.lib().yo_stub_key(b.ctypes.data_as(ctypes.POINTER(ctypes.c_int8)), n * m))


def hashed_form(board, n, m, seed):
    """The form random-form evaluation gives `board` under engine seed `seed`."""
    fs = forms(n, m)
    return fs[mix64(stub_key(board, n, m) ^ (seed & MASK64)) % len(fs)]


def average(outs):
    """fp32 mean over forms in ascending form order: ((o0 + o1) + o2) ... then x 1/F (a power of two: exact)."""
    s = np.asarray(outs[0], np.float32).copy()
    for o in outs[1:]:
        s = (s + np.asarray(o, np.float32)).astype(np.float32)
    return (s * np.float32(1.0 / len(outs))).astype(np.float32)
