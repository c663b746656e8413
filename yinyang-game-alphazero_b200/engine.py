"""Thin Python binding over the C ABI: device buffers come from torch, every computation is a CUDA kernel
of ``libyinyang_b200.so``.  Nothing here computes on the CPU; without a CUDA device the calls raise.

Device-tensor API (inputs already resident in HBM):
  legal_mask / step / ended / env_step / random_playout   -- batched rules (yin_yang_game.py:39-110)
  Engine.search / evaluate / selfplay_run                  -- mcts.py:275-343, neural_network.py:125-154,
                                                              self_play.py:72-192
Host-buffer API (numpy in, numpy out, copies inside): the ``*_host`` functions and ``Engine.search_host``.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, bitboard, weights as _weights

RULE_ROWCOL = 1
EVAL_STUB, EVAL_NN, EVAL_EXTERNAL = 0, 1, 2
MODE_SEARCH_AS_BLACK = 1
MODE_STEP_KERNELS = 2
MODE_EVAL_RANDOM_FORM = 4
MODE_EVAL_AVERAGE_FORMS = 8
# eval_symmetry -> mode_flags: evaluate every leaf as it is, in one form hashed from (seed, position), or averaged over all
# dihedral forms (include/yinyang_b200.h, YY_MODE_EVAL_*)
EVAL_SYMMETRY = {"none": 0, "random": MODE_EVAL_RANDOM_FORM, "average": MODE_EVAL_AVERAGE_FORMS}


def symmetry_forms(rows, cols):
    """The dihedral forms that keep a rows x cols board's shape, in augment_sample's order (0 identity, 1-3 rot90 x1/x2/x3,
    4 flip left-right, 5 flip up-down, 6 transpose, 7 anti-transpose)."""
    return list(range(8)) if rows == cols else [0, 2, 4, 5]
RESULT_DRAW_CODE = 2
DRAW_VALUE = 0.0001  # yin_yang_game.py:107


_cuda_seen = False


def _require_cuda():
    global _cuda_seen
    if _cuda_seen:                               # a device that was there stays there: ask once, not on every call
        return
    if not torch.cuda.is_available() or _lib.lib().yy_device_count() == 0:
        raise _lib.YinYangError("no CUDA device: the B200 engine has no CPU fallback")
    _cuda_seen = True


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def result_from_code(code):
    """YY_RESULT_* -> the reference's getGameEnded return value (0 / 1 / -1 / 0.0001)."""
    code = np.asarray(code)
    out = code.astype(np.float64)
    out[code == RESULT_DRAW_CODE] = DRAW_VALUE
    return out


# ------------------------------------------------------------------------------------------------ rules (device)
def _check_boards(black, white, players):
    assert black.is_cuda and white.is_cuda and players.is_cuda
    assert black.dtype == torch.int64 or black.dtype == torch.uint64
    assert players.dtype == torch.int8
    assert black.is_contiguous() and white.is_contiguous() and players.is_contiguous()


def legal_mask(black, white, players, rows, cols, rule_flags=0, out=None):
    """getValidMoves for every board: returns mask words int64[B, W] (bit a = action a legal)."""
    _require_cuda(); _check_boards(black, white, players)
    if out is None:
        out = torch.empty_like(black)
    _lib.check(_lib.lib().yy_legal_mask(rows, cols, rule_flags, _ptr(black), _ptr(white), _ptr(players), _ptr(out),
                                        players.numel(), _stream()))
    return out


def step(black, white, players, actions, rows, cols, rule_flags=0):
    """getNextState in place (illegal action = silent no-op; the turn passes either way)."""
    _require_cuda(); _check_boards(black, white, players)
    assert actions.dtype == torch.int32 and actions.is_cuda
    _lib.check(_lib.lib().yy_step(rows, cols, rule_flags, _ptr(black), _ptr(white), _ptr(players), _ptr(actions),
                                  players.numel(), _stream()))


def ended(black, white, players, rows, cols, rule_flags=0, out=None):
    """getGameEnded codes int8[B] (0 ongoing, 1 win, -1 loss, 2 draw) from players' perspective."""
    _require_cuda(); _check_boards(black, white, players)
    if out is None:
        out = torch.empty_like(players)
    _lib.check(_lib.lib().yy_ended(rows, cols, rule_flags, _ptr(black), _ptr(white), _ptr(players), _ptr(out),
                                   players.numel(), _stream()))
    return out


def env_step(black, white, players, actions, rows, cols, rule_flags=0, out_mask=None, out_result=None):
    """One fused environment step (mask of the side to move, apply, terminal code of the successor). In place."""
    _require_cuda(); _check_boards(black, white, players)
    if out_mask is None:
        out_mask = torch.empty_like(black)
    if out_result is None:
        out_result = torch.empty_like(players)
    _lib.check(_lib.lib().yy_env_step(rows, cols, rule_flags, _ptr(black), _ptr(white), _ptr(players), _ptr(actions),
                                      _ptr(out_mask), _ptr(out_result), players.numel(), _stream()))
    return out_mask, out_result


def augment_samples(black, white, rows, cols, counts=None, policy=None, values=None, out=None, forms=8):
    """Replay records -> training tensors with the reference's 8-fold augmentation (yy_augment_samples; replaces
    data_utils.create_dataset_from_games).  Device tensors in: black/white int64[N,W], counts int16/uint16[N,A] (visit
    counts) or policy float32[N,A], values float32[N] (optional).  Returns device tensors
    (planes float32[8N,5,n,m], policy float32[8N,A], values float32[8N] or None); sample 8r+f = form f of record r.
    ``out`` = a previous call's result tuple of the same sizes: written in place (no allocation of the 12 KB per record)."""
    _require_cuda()
    if (counts is None) == (policy is None):
        raise ValueError("give exactly one of counts / policy")
    n = black.shape[0]
    A = rows * cols
    dev = black.device
    assert forms in (1, 8)        # 1: no augmentation (yy_dataset_samples, any board shape); 8: the reference's 8 forms
    if out is not None:
        planes, pol, vals = out
        assert planes.is_contiguous() and pol.is_contiguous() and planes.dtype == pol.dtype == torch.float32
        assert planes.numel() == forms * n * 5 * A and pol.numel() == forms * n * A and planes.device == pol.device == dev
        assert (vals is None) == (values is None) and (vals is None or (vals.numel() == forms * n and vals.dtype == torch.float32))
    else:
        planes = torch.empty((forms * n, 5, rows, cols), dtype=torch.float32, device=dev)
        pol = torch.empty((forms * n, A), dtype=torch.float32, device=dev)
        vals = torch.empty(forms * n, dtype=torch.float32, device=dev) if values is not None else None
    if counts is not None:
        counts = counts.contiguous()
        assert counts.element_size() == 2 and counts.numel() == n * A
    if policy is not None:
        policy = policy.to(torch.float32).contiguous()
        assert policy.numel() == n * A
    if values is not None:
        values = values.to(torch.float32).contiguous()
    fn = _lib.lib().yy_augment_samples if forms == 8 else _lib.lib().yy_dataset_samples
    _lib.check(fn(rows, cols, _ptr(black), _ptr(white), _ptr(counts), _ptr(policy), _ptr(values),
                  n, _ptr(planes), _ptr(pol), _ptr(vals), _stream()))
    return planes, pol, vals


def augment_samples_host(boards, rows, cols, counts=None, policy=None, values=None, forms=8):
    """numpy in / numpy out variant of augment_samples (H2D + kernel + D2H)."""
    _require_cuda()
    b, w = bitboard.pack_boards(boards, rows, cols)
    c = _to_dev(np.ascontiguousarray(counts, dtype=np.uint16).view(np.int16), torch.int16) if counts is not None else None
    p = _to_dev(np.ascontiguousarray(policy, dtype=np.float32), torch.float32) if policy is not None else None
    v = _to_dev(np.ascontiguousarray(values, dtype=np.float64).astype(np.float32), torch.float32) if values is not None else None
    planes, pol, vals = augment_samples(_to_dev(b, torch.int64), _to_dev(w, torch.int64), rows, cols, counts=c, policy=p, values=v, forms=forms)
    return planes.cpu().numpy(), pol.cpu().numpy(), (vals.cpu().numpy() if vals is not None else None)


def random_playout(count, plies, rows, cols, seed=0xC0FFEE, rule_flags=0, device="cuda"):
    """Synthetic boards: board i = empty board advanced by plies[i] uniformly random legal plies."""
    _require_cuda()
    W = bitboard.words_for(rows, cols)
    black = torch.empty((count, W), dtype=torch.int64, device=device)
    white = torch.empty((count, W), dtype=torch.int64, device=device)
    players = torch.empty(count, dtype=torch.int8, device=device)
    plies = plies.to(device=device, dtype=torch.int32).contiguous()
    _lib.check(_lib.lib().yy_random_playout(rows, cols, rule_flags, ctypes.c_uint64(seed), _ptr(plies), _ptr(black),
                                            _ptr(white), _ptr(players), count, _stream()))
    return black, white, players


# ------------------------------------------------------------------------------------------------ rules (host buffers)
def _to_dev(a, dtype):
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint64:
        a = a.view(np.int64)
    t = torch.from_numpy(a)
    return t.pin_memory().to("cuda", non_blocking=True).view(dtype) if t.numel() else t.to("cuda").view(dtype)


def _to_host(*tensors):
    """Device tensors -> numpy arrays through pinned buffers of torch's caching host allocator: the copies run at the
    PCIe rate on the current stream (no pageable staging, no first-touch page faults), one synchronisation for all.
    Each array owns its buffer (returned to the allocator's cache when the array dies)."""
    hosts = []
    for t in tensors:
        if t is None or t.numel() == 0:
            hosts.append(None if t is None else t.cpu())
            continue
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t, non_blocking=True)
        hosts.append(h)
    torch.cuda.current_stream().synchronize()
    return tuple(None if h is None else h.numpy() for h in hosts)


_DEVICE_PACK_MIN = 512      # from this many boards on, the int8 <-> bitboard conversion runs on the GPU


def pack_boards_dev(boards, rows, cols):
    """numpy int8[B,n,m] -> device bitboards (black int64[B,W], white int64[B,W]); the packing itself on the GPU."""
    B, W = int(np.asarray(boards).shape[0]), bitboard.words_for(rows, cols)
    bd_i8 = _to_dev(np.ascontiguousarray(boards, dtype=np.int8).reshape(B, rows * cols), torch.int8)
    black = torch.empty((B, W), dtype=torch.int64, device="cuda"); white = torch.empty_like(black)
    _lib.check(_lib.lib().yy_pack_boards(rows, cols, _ptr(bd_i8), _ptr(black), _ptr(white), B, _stream()))
    return black, white


def unpack_boards_dev(rows, cols, black=None, white=None, mask=None):
    """Device bitboards -> (numpy int8[B,n,m] boards or None, numpy uint8[B,A] mask bits or None); unpacked on the GPU."""
    ref = black if black is not None else mask
    B, A = ref.shape[0], rows * cols
    ob = torch.empty((B, A), dtype=torch.int8, device="cuda") if black is not None else None
    om = torch.empty((B, A), dtype=torch.uint8, device="cuda") if mask is not None else None
    _lib.check(_lib.lib().yy_unpack_boards(rows, cols, _ptr(black), _ptr(white), _ptr(mask), _ptr(ob), _ptr(om), B, _stream()))
    hb, hm = _to_host(ob, om)
    return (hb.reshape(B, rows, cols) if hb is not None else None, hm)


def _boards_to_dev(boards, rows, cols):
    if np.asarray(boards).shape[0] >= _DEVICE_PACK_MIN:
        return pack_boards_dev(boards, rows, cols)
    b, w = bitboard.pack_boards(boards, rows, cols)
    return _to_dev(b, torch.int64), _to_dev(w, torch.int64)


def legal_mask_host(boards, players, rows, cols, rule_flags=0):
    """numpy int8[B,n,m] boards, int8[B] players -> uint8[B, A] masks.  H2D + kernel + D2H."""
    _require_cuda()
    bd, wd = _boards_to_dev(boards, rows, cols)
    mask = legal_mask(bd, wd, _to_dev(np.asarray(players, np.int8), torch.int8), rows, cols, rule_flags)
    if mask.shape[0] >= _DEVICE_PACK_MIN:
        return unpack_boards_dev(rows, cols, mask=mask)[1]
    return bitboard.unpack_bits(mask.cpu().numpy().view(np.uint64), rows, cols)


def env_step_host(boards, players, actions, rows, cols, rule_flags=0):
    """Host-buffer env step: returns (masks uint8[B,A], boards' int8[B,n,m], players' int8[B], results f64[B])."""
    _require_cuda()
    bd, wd = _boards_to_dev(boards, rows, cols)
    pd = _to_dev(np.asarray(players, np.int8), torch.int8)
    ad = _to_dev(np.asarray(actions, np.int32), torch.int32)
    mask, res = env_step(bd, wd, pd, ad, rows, cols, rule_flags)
    if mask.shape[0] >= _DEVICE_PACK_MIN:
        nb, bits = unpack_boards_dev(rows, cols, bd, wd, mask)
    else:
        bits = bitboard.unpack_bits(mask.cpu().numpy().view(np.uint64), rows, cols)
        nb = bitboard.unpack_boards(bd.cpu().numpy().view(np.uint64), wd.cpu().numpy().view(np.uint64), rows, cols)
    hp, hr = _to_host(pd, res)
    return bits, nb, hp, result_from_code(hr)


def env_step_host_packed(black, white, players, actions, rows, cols, rule_flags=0):
    """Host-buffer env step on PACKED boards (the layout of include/yinyang_b200.h: uint64[B, W] per colour): numpy in,
    numpy out -- (mask words uint64[B,W], black' uint64[B,W], white' uint64[B,W], players' int8[B], result codes int8[B]).
    21 bytes in and 26 out per 8x8 board instead of the 69 / 193 of the int8-array entry point."""
    _require_cuda()
    bd, wd = _to_dev(np.ascontiguousarray(black, dtype=np.uint64), torch.int64), _to_dev(np.ascontiguousarray(white, dtype=np.uint64), torch.int64)
    pd = _to_dev(np.asarray(players, np.int8), torch.int8)
    ad = _to_dev(np.asarray(actions, np.int32), torch.int32)
    mask, res = env_step(bd, wd, pd, ad, rows, cols, rule_flags)
    hm, hb, hw, hp, hr = _to_host(mask, bd, wd, pd, res)
    return hm.view(np.uint64), hb.view(np.uint64), hw.view(np.uint64), hp, hr


def next_state_host(boards, players, actions, rows, cols, rule_flags=0):
    _require_cuda()
    b, w = bitboard.pack_boards(boards, rows, cols)
    bd, wd = _to_dev(b, torch.int64), _to_dev(w, torch.int64)
    pd = _to_dev(np.asarray(players, np.int8), torch.int8)
    step(bd, wd, pd, _to_dev(np.asarray(actions, np.int32), torch.int32), rows, cols, rule_flags)
    return (bitboard.unpack_boards(bd.cpu().numpy().view(np.uint64), wd.cpu().numpy().view(np.uint64), rows, cols),
            pd.cpu().numpy())


def ended_host(boards, players, rows, cols, rule_flags=0):
    _require_cuda()
    b, w = bitboard.pack_boards(boards, rows, cols)
    code = ended(_to_dev(b, torch.int64), _to_dev(w, torch.int64), _to_dev(np.asarray(players, np.int8), torch.int8),
                 rows, cols, rule_flags)
    return result_from_code(code.cpu().numpy())


# ------------------------------------------------------------------------------------------------ engine
def device_image(image, device):
    """A packed weight image (numpy uint8, weights.pack_state_dict) -> a 256-byte aligned uint8 view on the device."""
    with torch.cuda.device(device):
        buf = torch.zeros(image.size + 256, dtype=torch.uint8, device=torch.device("cuda", device))
        off = (-buf.data_ptr()) & 255
        view = buf[off: off + image.size]
        view.copy_(torch.from_numpy(image))
        torch.cuda.synchronize()
    return view


@dataclass
class Stats:
    moves: int
    evals: int
    games_finished: int
    examples: int
    sims: int
    overflow: int
    max_depth: int
    tower_evals: int = 0


class Engine:
    """n_games concurrent MCTS trees + evaluator + self-play slots on one GPU (yy_engine)."""

    def __init__(self, rows=8, cols=8, n_games=1, n_sims=800, evaluator="stub", cpuct=1.0, rule_flags=0,
                 search_as_black=True, edges_per_game=0, dirichlet_alpha=0.3, dirichlet_epsilon=0.25,
                 temperature_threshold=10, seed=0, replay_capacity=0, state_dict=None, nn_channels=128, nn_blocks=10,
                 device=None, leaves_per_step=1, step_kernels=False, descents_per_step=0, eval_symmetry="none",
                 weight_image=None):
        if eval_symmetry not in EVAL_SYMMETRY:
            raise ValueError(f"eval_symmetry must be one of {sorted(EVAL_SYMMETRY)}, not {eval_symmetry!r}")
        if eval_symmetry != "none" and evaluator != "nn":
            raise ValueError("eval_symmetry needs evaluator='nn'")
        _require_cuda()
        self.L = _lib.lib()
        self.rows, self.cols, self.A, self.W = rows, cols, rows * cols, bitboard.words_for(rows, cols)
        self.n_games, self.n_sims = n_games, n_sims
        self.leaves_per_step = max(1, int(leaves_per_step))
        self.n_slots = n_games * self.leaves_per_step
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.tdev = torch.device("cuda", self.device)
        ev = {"stub": EVAL_STUB, "nn": EVAL_NN, "external": EVAL_EXTERNAL}[evaluator]
        self.evaluator = evaluator
        self.eval_symmetry = eval_symmetry
        if evaluator == "nn" and weight_image is None:      # (a packed image comes with nn_channels / nn_blocks)
            if state_dict is None:
                raise ValueError("evaluator='nn' needs a reference state_dict / checkpoint dict")
            sd = state_dict["state_dict"] if "state_dict" in state_dict else state_dict
            nn_channels, nn_blocks = _weights.infer_arch(sd)
        if replay_capacity <= 0:
            replay_capacity = max(1, n_games * (self.A + 8))
        self.cfg = _lib.EngineConfig(rows=rows, cols=cols, n_games=n_games, n_sims=n_sims, rule_flags=rule_flags,
                                     mode_flags=(MODE_SEARCH_AS_BLACK if search_as_black else 0) | (MODE_STEP_KERNELS if step_kernels else 0)
                                     | EVAL_SYMMETRY[eval_symmetry], evaluator=ev,
                                     edges_per_game=edges_per_game, temperature_threshold=temperature_threshold,
                                     replay_capacity=replay_capacity, nn_channels=nn_channels, nn_blocks=nn_blocks,
                                     device=self.device, leaves_per_step=self.leaves_per_step, cpuct=cpuct, descents_per_step=int(descents_per_step),
                                     dirichlet_alpha=dirichlet_alpha,
                                     dirichlet_epsilon=dirichlet_epsilon, seed=seed)
        need = self.L.yy_engine_workspace_bytes(ctypes.byref(self.cfg))
        if need < 0:
            _lib.check(int(need))
        with torch.cuda.device(self.device):
            self.workspace = torch.zeros(int(need) + 256, dtype=torch.uint8, device=self.tdev)
            base = self.workspace.data_ptr()
            self._ws_ptr = (base + 255) & ~255
            torch.cuda.synchronize()
            self.handle = self.L.yy_engine_create(ctypes.byref(self.cfg), ctypes.c_void_p(self._ws_ptr), int(need))
        if not self.handle:
            _lib.check(-1)
        self.weight_image = None
        if evaluator == "nn" and weight_image is not None:
            self.load_weight_image(weight_image)
        elif evaluator == "nn":
            self.load_state_dict(state_dict)
        self.replay_capacity = replay_capacity
        self.workspace_bytes = int(need)

    # -- lifetime
    def close(self):
        if getattr(self, "handle", None):
            torch.cuda.synchronize(self.device)
            self.L.yy_engine_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- weights (yy_engine_load_weights)
    def load_state_dict(self, state_dict):
        img = _weights.pack_state_dict(state_dict, self.rows, self.cols)
        view = device_image(img, self.device)
        self.weight_image = view
        _lib.check(self.L.yy_engine_load_weights(self.handle, _ptr(view), img.size))

    def load_weight_image(self, image_u8: torch.Tensor):
        """Adopt an already-packed device image (e.g. one received over an NCCL broadcast)."""
        assert image_u8.is_cuda and image_u8.dtype == torch.uint8 and image_u8.data_ptr() % 256 == 0
        self.weight_image = image_u8
        _lib.check(self.L.yy_engine_load_weights(self.handle, _ptr(image_u8), image_u8.numel()))

    # -- search (MCTS.search for all games)
    def search(self, black, white, players, noise=None, noise_mask=None, out_counts=None):
        """Device tensors in, root visit counts int32[n_games, A] out (mcts.py:168-181)."""
        _check_boards(black, white, players)
        assert players.numel() == self.n_games
        if out_counts is None:
            out_counts = torch.empty((self.n_games, self.A), dtype=torch.int32, device=self.tdev)
        _lib.check(self.L.yy_search(self.handle, _ptr(black), _ptr(white), _ptr(players), _ptr(noise), _ptr(noise_mask),
                                    _ptr(out_counts), _stream()))
        return out_counts

    def search_host(self, boards, players, noise=None):
        """numpy int8[n_games,n,m] boards (or a (black, white) pair of packed uint64[n_games, W] arrays) + players ->
        (counts int32[n_games,A], child value sums f32)."""
        b, w = boards if isinstance(boards, tuple) else bitboard.pack_boards(boards, self.rows, self.cols)
        bd, wd = _to_dev(b, torch.int64), _to_dev(w, torch.int64)
        pd = _to_dev(np.asarray(players, np.int8), torch.int8)
        nz = nm = None
        if noise is not None:
            full = np.zeros((self.n_games, self.A), dtype=np.float64)
            mask = np.zeros(self.n_games, dtype=np.uint8)
            for g, nzg in enumerate(noise):
                if nzg is not None and len(nzg):
                    full[g, : len(nzg)] = nzg
                    mask[g] = 1
            nz, nm = _to_dev(full, torch.float64), _to_dev(mask, torch.uint8)
        counts = self.search(bd, wd, pd, nz, nm)
        cw = torch.empty((self.n_games, self.A), dtype=torch.float32, device=self.tdev)
        c2 = torch.empty_like(counts)
        _lib.check(self.L.yy_search_counts(self.handle, _ptr(c2), _ptr(cw), _stream()))
        return _to_host(counts, cw)

    # -- external-evaluator stepping
    def search_begin(self, black, white, players, noise=None, noise_mask=None):
        _lib.check(self.L.yy_search_begin(self.handle, _ptr(black), _ptr(white), _ptr(players), _ptr(noise),
                                          _ptr(noise_mask), _stream()))

    def search_advance(self, priors=None, values=None) -> int:
        active = ctypes.c_int32(0)
        _lib.check(self.L.yy_search_advance(self.handle, _ptr(priors), _ptr(values), ctypes.byref(active), _stream()))
        return int(active.value)

    def leaf_batch(self):
        """(black int64[n_slots,W], white, active uint8[n_slots]) views of the pending leaf batch (slot = game*K + k)."""
        def view(ptr, n, dtype):
            off = ptr - self.workspace.data_ptr()
            return self.workspace[off: off + n].view(dtype)
        nb = self.n_slots * self.W * 8
        return (view(self.L.yy_engine_leaf_black(self.handle), nb, torch.int64).view(self.n_slots, self.W),
                view(self.L.yy_engine_leaf_white(self.handle), nb, torch.int64).view(self.n_slots, self.W),
                view(self.L.yy_engine_leaf_active(self.handle), self.n_slots, torch.uint8))

    def tree_host(self, game=0):
        """The whole search tree of one game as numpy arrays (yy_engine_tree_view): dict(n_nodes, edge_base, n_edges, player,
        flags, value, black, white per node; N, W, P, child (node id or -1), child_flags, action per edge slot)."""
        v = _lib.TreeView()
        _lib.check(self.L.yy_engine_tree_view(self.handle, ctypes.byref(v)))
        base = self.workspace.data_ptr()

        def grab(ptr, first, count, dtype, itemsize):
            off = ptr - base + first * itemsize
            return self.workspace[off: off + count * itemsize].view(dtype)
        nn = int(grab(v.n_nodes, game, 1, torch.int32, 4).item())
        ne = int(grab(v.n_edges_used, game, 1, torch.int32, 4).item())
        n0, e0, W = game * v.max_nodes, game * v.edges_cap, v.W
        dev = {"edge_base": grab(v.node_edge_base, n0, nn, torch.int32, 4), "n_edges": grab(v.node_n_edges, n0, nn, torch.int16, 2),
               "player": grab(v.node_player, n0, nn, torch.int8, 1), "flags": grab(v.node_flags, n0, nn, torch.uint8, 1),
               "value": grab(v.node_value, n0, nn, torch.float32, 4),
               "black": grab(v.node_black, n0 * W, nn * W, torch.int64, 8), "white": grab(v.node_white, n0 * W, nn * W, torch.int64, 8),
               "N": grab(v.edge_N, e0, ne, torch.int32, 4), "W": grab(v.edge_W, e0, ne, torch.float32, 4),
               "P": grab(v.edge_P, e0, ne, torch.float32, 4), "meta": grab(v.edge_child_meta, e0, ne, torch.int64, 8),
               "action": grab(v.edge_action, e0, ne, torch.uint8, 1)}
        keys = sorted(dev)
        host = dict(zip(keys, _to_host(*[dev[k] for k in keys])))
        host = {k: (h if h is not None else np.zeros(0, dtype=np.int64)) for k, h in host.items()}
        meta = host.pop("meta").view(np.uint64)
        host["child"] = ((meta >> np.uint64(32)) & np.uint64(0xFFFF)).astype(np.int64) - 1
        host["child_flags"] = ((meta >> np.uint64(57)) & np.uint64(7)).astype(np.uint8)
        host["black"] = host["black"].view(np.uint64).reshape(nn, W); host["white"] = host["white"].view(np.uint64).reshape(nn, W)
        host["n_nodes"] = nn
        return host

    def search_counts(self):
        counts = torch.empty((self.n_games, self.A), dtype=torch.int32, device=self.tdev)
        cw = torch.empty((self.n_games, self.A), dtype=torch.float32, device=self.tdev)
        _lib.check(self.L.yy_search_counts(self.handle, _ptr(counts), _ptr(cw), _stream()))
        return counts, cw

    # -- evaluator on an arbitrary batch (batched predict)
    def evaluate(self, black, white, want_logits=False, form=None):
        """form=None: the engine's own eval_symmetry; an int: that dihedral form (symmetry_forms), outputs mapped back to
        the board's actions; "average": policy and value averaged over all forms (no logits)."""
        n = black.shape[0]
        policy = torch.empty((n, self.A), dtype=torch.float32, device=self.tdev)
        value = torch.empty(n, dtype=torch.float32, device=self.tdev)
        logits = torch.empty((n, self.A), dtype=torch.float32, device=self.tdev) if want_logits else None
        if form is None:
            _lib.check(self.L.yy_evaluate(self.handle, _ptr(black), _ptr(white), n, _ptr(policy), _ptr(value), _ptr(logits),
                                          _stream()))
        else:
            if form == "average":
                code = -1
            elif isinstance(form, (int, np.integer)) and not isinstance(form, bool) and 0 <= int(form) <= 7:
                code = int(form)
            else:
                raise ValueError(f"form must be None, 0..7 or 'average', not {form!r}")
            _lib.check(self.L.yy_evaluate_form(self.handle, _ptr(black), _ptr(white), n, code, _ptr(policy), _ptr(value),
                                               _ptr(logits), _stream()))
        return (policy, value, logits) if want_logits else (policy, value)

    def evaluate_host(self, boards, want_logits=False, form=None):
        b, w = bitboard.pack_boards(boards, self.rows, self.cols)
        out = self.evaluate(_to_dev(b, torch.int64), _to_dev(w, torch.int64), want_logits, form=form)
        return tuple(o.cpu().numpy() for o in out)

    # -- profiling of the dominant kernel
    def set_profiling(self, enable=True):
        _lib.check(self.L.yy_engine_set_profiling(self.handle, 1 if enable else 0))

    def get_profile(self):
        """-> dict(launches, ms, boards) of the tower kernel since set_profiling(True)."""
        l, b, ms = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_double(0)
        _lib.check(self.L.yy_engine_get_profile(self.handle, ctypes.byref(l), ctypes.byref(ms), ctypes.byref(b)))
        return {"launches": int(l.value), "ms": float(ms.value), "boards": int(b.value)}

    # -- self-play
    def selfplay_reset(self):
        _lib.check(self.L.yy_selfplay_reset(self.handle, _stream()))

    def selfplay_run(self, n_moves: int):
        """Asynchronous: enqueues n_moves full searches + moves per game slot on the current stream (one launch of the
        persistent kernel; the slots advance independently)."""
        _lib.check(self.L.yy_selfplay_run(self.handle, int(n_moves), _stream()))

    def selfplay_advance(self, iterations: int):
        """Rolling self-play: `iterations` evaluation steps (one leaf per game slot per step) in one launch; searches in
        progress continue with the next call.  Completed moves / games: stats()."""
        _lib.check(self.L.yy_selfplay_advance(self.handle, int(iterations), _stream()))

    def selfplay_set_quota(self, total_games):
        """At most total_games games are started since the last reset (None / negative: unlimited)."""
        _lib.check(self.L.yy_selfplay_set_quota(self.handle, -1 if total_games is None else int(total_games)))

    def selfplay_set_playout_cap(self, full_prob=1.0, fast_sims=None):
        """Playout cap randomisation of self-play (yy_selfplay_set_playout_cap): each move is a full search (n_sims, noise at
        ply 0, recorded) with probability full_prob -- a hash of (seed, game serial, ply) decides -- otherwise a fast search
        of fast_sims simulations (None: n_sims) that adds no noise and no replay record.  full_prob=1 turns it off.  Applies
        from the next search root each slot prepares; search() ignores it."""
        fast = self.n_sims if fast_sims is None else int(fast_sims)
        _lib.check(self.L.yy_selfplay_set_playout_cap(self.handle, float(full_prob), fast))

    def selfplay_set_random_stream(self, uniforms=None, noise=None):
        """Recorded random stream (yy_selfplay_set_random_stream): uniforms float64[n_games, n_plies], noise float64[n_games, A]
        (numpy or device tensors).  None, None restores Philox."""
        def dev(x):
            if x is None:
                return None
            t = x if torch.is_tensor(x) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64))
            return t.to(device=self.tdev, dtype=torch.float64).contiguous()
        u, z = dev(uniforms), dev(noise)
        if z is not None:
            assert z.shape[1] == self.A
        ng = int(u.shape[0]) if u is not None else (int(z.shape[0]) if z is not None else 0)
        if u is not None and z is not None:
            assert u.shape[0] == z.shape[0]
        npl = int(u.shape[1]) if u is not None else (1 if z is not None else 0)
        self._random_stream = (u, z)                                   # the engine keeps the pointers: keep them alive
        _lib.check(self.L.yy_selfplay_set_random_stream(self.handle, _ptr(u), _ptr(z), ng, npl))

    # -- arena (yy_arena_run)
    def arena_run(self, image_b, start_black, start_white, start_player, a_plays_black, max_plies):
        """n_games / 2 arena games, model A = the loaded weights (slots [0, G)), model B = image_b (a packed device image of
        the same network shape, 256-byte aligned; slots [G, 2G)).  Device tensors in: start boards int64[G, W], players to
        move int8[G], a_plays_black uint8/bool[G].  Every move is the temperature-0 choice of a noise-free search; a game
        ends on a terminal position or after max_plies plies.  Returns device tensors (codes int8[G]: YY_RESULT_* of the
        player to move after the last move, 0 at the ply cap; plies int32[G]).  Leaves the self-play slots reset."""
        G = self.n_games // 2
        _check_boards(start_black, start_white, start_player)
        assert image_b.is_cuda and image_b.dtype == torch.uint8 and image_b.is_contiguous()
        assert start_player.numel() == G and start_black.shape[0] == G and a_plays_black.numel() == G
        ab = a_plays_black.to(device=self.tdev, dtype=torch.uint8).contiguous()
        codes = torch.empty(G, dtype=torch.int8, device=self.tdev)
        plies = torch.empty(G, dtype=torch.int32, device=self.tdev)
        _lib.check(self.L.yy_arena_run(self.handle, _ptr(image_b), image_b.numel(), _ptr(start_black), _ptr(start_white),
                                       _ptr(start_player), _ptr(ab), int(max_plies), _ptr(codes), _ptr(plies), _stream()))
        return codes, plies

    def stats(self) -> Stats:
        s = _lib.SelfPlayStats()
        _lib.check(self.L.yy_selfplay_get_stats(self.handle, ctypes.byref(s), _stream()))
        return Stats(s.moves, s.evals, s.games_finished, s.examples, s.sims, s.overflow, s.max_depth, s.tower_evals)

    # -- replay ring: device views and windows
    def replay_views(self):
        """Device views (no copy) over the WHOLE replay ring (replay_capacity rows; row = record index % capacity):
        black / white int64[cap, W], counts int16[cap, A] (uint16 bit pattern), game_serial int32[cap], ply int16[cap],
        player int8[cap], and the results table int8[results_capacity] (code of game s at [s % results_capacity])."""
        if getattr(self, "_rviews", None) is None:
            v = _lib.ReplayView()
            _lib.check(self.L.yy_selfplay_replay(self.handle, ctypes.byref(v)))
            base, cap = self.workspace.data_ptr(), self.replay_capacity

            def view(ptr, nbytes, dtype, shape):
                return self.workspace[ptr - base: ptr - base + nbytes].view(dtype).view(shape)
            self._rviews = {"black": view(v.black, cap * self.W * 8, torch.int64, (cap, self.W)),
                            "white": view(v.white, cap * self.W * 8, torch.int64, (cap, self.W)),
                            "counts": view(v.counts, cap * self.A * 2, torch.int16, (cap, self.A)),
                            "game_serial": view(v.game_serial, cap * 4, torch.int32, (cap,)),
                            "ply": view(v.ply, cap * 2, torch.int16, (cap,)),
                            "player": view(v.player, cap, torch.int8, (cap,)),
                            "results": view(v.results, v.results_capacity, torch.int8, (v.results_capacity,))}
            self.results_capacity = int(v.results_capacity)
        return self._rviews

    def replay_window_dev(self, start, stop):
        """Device tensors (views when the window does not wrap, else copies) of the records with global indices
        [start, stop), oldest first; stop - start <= replay_capacity."""
        rv, cap = self.replay_views(), self.replay_capacity
        n = stop - start
        assert 0 <= n <= cap
        lo, hi = start % cap, start % cap + n
        keys = ("black", "white", "counts", "game_serial", "ply", "player")
        if hi <= cap:
            return {k: rv[k][lo:hi] for k in keys}
        return {k: torch.cat([rv[k][lo:], rv[k][: hi - cap]], dim=0) for k in keys}

    def replay_window(self, start, stop):
        """The same window on the host (numpy, through pinned buffers, one synchronisation)."""
        w = self.replay_window_dev(start, stop)
        keys = sorted(w)
        host = _to_host(*[w[k] for k in keys])
        out = {k: (h if h is not None else np.zeros((0,) + tuple(w[k].shape[1:]), dtype=np.int64)) for k, h in zip(keys, host)}
        out["black"] = out["black"].view(np.uint64); out["white"] = out["white"].view(np.uint64)
        out["counts"] = out["counts"].view(np.uint16)
        return out

    def stats_view(self):
        """Device view int64[7] of the live counters (moves, evals, games_finished, examples, sims, overflow | max_depth << 32,
        tower_evals): copy it on the launching stream for a snapshot that is ordered with the self-play launches."""
        ptr = self.L.yy_selfplay_stats_dev(self.handle)
        off = ptr - self.workspace.data_ptr()
        return self.workspace[off: off + 56].view(torch.int64)

    def replay(self):
        """Copies the replay ring to the host: dict(boards int8[N,n,m], counts uint16[N,A], pi float64[N,A],
        game_serial, ply, player, z float64[N] (NaN while the game is unfinished))."""
        st = self.stats()
        n = min(st.examples, self.replay_capacity)
        v = _lib.ReplayView()
        _lib.check(self.L.yy_selfplay_replay(self.handle, ctypes.byref(v)))
        base = self.workspace.data_ptr()

        def view(ptr, nbytes):
            return self.workspace[ptr - base: ptr - base + nbytes]
        bl = view(v.black, n * self.W * 8).cpu().numpy().view(np.uint64).reshape(n, self.W)
        wh = view(v.white, n * self.W * 8).cpu().numpy().view(np.uint64).reshape(n, self.W)
        counts = view(v.counts, n * self.A * 2).cpu().numpy().view(np.uint16).reshape(n, self.A)
        serial = view(v.game_serial, n * 4).cpu().numpy().view(np.int32)
        ply = view(v.ply, n * 2).cpu().numpy().view(np.int16)
        player = view(v.player, n).cpu().numpy().view(np.int8)
        results = view(v.results, v.results_capacity).cpu().numpy().view(np.int8)
        tot = counts.sum(axis=1, keepdims=True).astype(np.float64)
        pi = np.where(tot > 0, counts.astype(np.float64) / np.maximum(tot, 1), 1.0 / self.A)  # mcts.py:209-213
        finished = np.zeros(v.results_capacity, dtype=bool)
        z = np.full(n, np.nan)
        code = results[serial % v.results_capacity]
        z = np.where(code == 0, np.nan, result_from_code(code))
        return {"boards": bitboard.unpack_boards(bl, wh, self.rows, self.cols), "counts": counts, "pi": pi,
                "game_serial": serial, "ply": ply, "player": player, "z": z, "finished": ~np.isnan(z)}

    def live_boards(self):
        nb = self.n_games * self.W * 8
        base = self.workspace.data_ptr()
        pb, pw, pp = (self.L.yy_engine_game_black(self.handle), self.L.yy_engine_game_white(self.handle),
                      self.L.yy_engine_game_player(self.handle))
        bl = self.workspace[pb - base: pb - base + nb].cpu().numpy().view(np.uint64).reshape(self.n_games, self.W)
        wh = self.workspace[pw - base: pw - base + nb].cpu().numpy().view(np.uint64).reshape(self.n_games, self.W)
        pl = self.workspace[pp - base: pp - base + self.n_games].cpu().numpy().view(np.int8)
        return bitboard.unpack_boards(bl, wh, self.rows, self.cols), pl
