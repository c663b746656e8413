"""Integer-valued networks on which the bf16 tower is exact (test infrastructure).

Every weight is a small integer (value_fc2: a multiple of 2^-8), every BatchNorm folds to "+ beta" with beta in
{-1, 0, 1}, and the draw is checked on the positions under test: every intermediate is an integer, every ReLU output
lies in [0, 255] and every accumulator below 2^24 in magnitude.  Then bf16 rounding is the identity on weights and
activations and fp32 accumulation is exact in any order, so the kernel must reproduce the float64 reference's logits
bit for bit, at any depth, width and board geometry.

Also the geometry classes of the network kernel: the code paths that a board size selects in yy_tower.cuh /
yy_fused.cu (position layout, FC-head tiling, clamped group size), and one representative board per class.
"""
import ctypes
import itertools

import numpy as np

BN_EPS = 1e-5
BN_VAR = 1.0 - BN_EPS     # weights._fold: 1 / sqrt(float32(BN_VAR) + eps) = 1 + 7e-9, which is exactly 1.0 in float32
MAX_ACT = 255             # ReLU outputs must be bf16-exact integers
MAX_ACC = 1 << 24         # fp32 sums of integers are exact below this

# Boards the GPU tests run, one or more per geometry class (see geometry_class).  The class-coverage test in
# test_host_logic.py fails when a class of the 500 supported geometries has none here.
# (rows, cols, channels, blocks): a 128 x 10 net for one geometry of each of the five position layouts.
REPRESENTATIVES = [
    (8, 8, 128, 10), (6, 6, 128, 10), (16, 16, 128, 10), (10, 8, 128, 10), (12, 12, 128, 10),
    (5, 7, 64, 2), (4, 8, 32, 2), (16, 8, 64, 1), (32, 8, 128, 2), (13, 11, 128, 1), (10, 10, 64, 2),
    (9, 11, 32, 1), (11, 22, 128, 2), (7, 7, 64, 2), (3, 3, 32, 2), (2, 2, 128, 1), (7, 1, 32, 2), (1, 8, 64, 1),
    (8, 22, 128, 1), (7, 9, 32, 0), (1, 1, 64, 1), (8, 16, 128, 1), (15, 17, 32, 2), (12, 16, 64, 1),
    (17, 8, 128, 2), (24, 8, 32, 1), (25, 8, 64, 2), (5, 10, 128, 0), (5, 1, 64, 1), (6, 18, 32, 2),
    (5, 21, 128, 1), (3, 22, 64, 0), (10, 20, 64, 1), (7, 19, 128, 2),
]


# ------------------------------------------------------------------------------------------------ geometry classes
def tower_classes(lib, rows, cols):
    """The product headers' choices for a board (tests/_host/tower_layout_check.cu yyh_tower_classes), or None when
    the network kernel does not accept the board."""
    out = (ctypes.c_int * 9)()
    if lib.yyh_tower_classes(rows, cols, out) != 0:
        return None
    keys = ["layout", "Gb_raw", "Gb", "T", "Tp", "n_panels", "KS", "Rp_last", "batch"]
    return dict(zip(keys, [int(v) for v in out]))


def geometry_class(c):
    """Code-path class of a board: layout, policy M tiles, multi-panel heads, partial last K panel, merged policy
    slots (last policy tile <= 64 rows: two K stages per weight slot), odd stage count, group size clamped to FC_N."""
    return (c["layout"], c["Tp"], c["n_panels"] > 1, c["KS"] % 32 != 0, c["Rp_last"] <= 64, c["KS"] % 2 == 1,
            c["Gb_raw"] > c["Gb"])


def supported_geometries(lib):
    return [(r, c) for r in range(1, 33) for c in range(1, 33) if r * c <= 256 and tower_classes(lib, r, c) is not None]


# ------------------------------------------------------------------------------------------------ the network
def _pm1(rng, rows, cols, plus, minus):
    """[rows][cols] with `plus` entries +1 and `minus` entries -1 per row, at distinct random columns."""
    w = np.zeros((rows, cols))
    for r in range(rows):
        idx = rng.choice(cols, size=plus + minus, replace=False)
        w[r, idx[:plus]], w[r, idx[plus:]] = 1.0, -1.0
    return w


def _draw(n, m, channels, blocks, seed):
    """Integer weights of one draw: dict of float64 arrays keyed like oracle/port.py build_net's state_dict."""
    rng = np.random.default_rng(seed)
    C, A = channels, n * m
    w = {}

    def conv_bn(name, bn, wt):
        w[name + ".weight"] = wt
        w[name + ".bias"] = np.zeros(wt.shape[0])
        w[bn + ".weight"] = np.ones(wt.shape[0])
        w[bn + ".bias"] = rng.integers(-1, 2, wt.shape[0]).astype(np.float64)
        w[bn + ".running_mean"] = np.zeros(wt.shape[0])
        w[bn + ".running_var"] = np.full(wt.shape[0], BN_VAR)

    # stem: planes 0-2 (one-hot cells); the fill planes 3 / 4 only where m * rf (n * cf) is exact in bf16
    stem = np.zeros((C, 5, 3, 3))
    stem[:, :3] = _pm1(rng, C, 27, 2, 1).reshape(C, 3, 3, 3)
    for plane, side in ((3, m), (4, n)):
        if side & (side - 1) == 0:
            taps = rng.integers(0, 9, C)
            sel = rng.random(C) < 1 / 16      # (a few channels, mostly negative: a row count is up to 32)
            stem[sel, plane, taps[sel] // 3, taps[sel] % 3] = side * np.where(rng.random(sel.sum()) < 0.75, -1.0, 1.0)
    conv_bn("conv1", "bn1", stem)
    for i in range(blocks):
        # conv1 balanced, conv2 leaning negative: the skip connection carries the block input, so a balanced conv2 would
        # let the activations grow geometrically with depth (measured: past 255 by block 7 of a 128 x 10 net)
        conv_bn(f"res_blocks.{i}.conv1", f"res_blocks.{i}.bn1", _pm1(rng, C, C * 9, 2, 2).reshape(C, C, 3, 3))
        conv_bn(f"res_blocks.{i}.conv2", f"res_blocks.{i}.bn2", _pm1(rng, C, C * 9, 1, 4).reshape(C, C, 3, 3))
    conv_bn("policy_conv", "policy_bn", _pm1(rng, 32, C, 2, 2).reshape(32, C, 1, 1))
    conv_bn("value_conv", "value_bn", _pm1(rng, 32, C, 2, 2).reshape(32, C, 1, 1))
    w["policy_fc.weight"] = _pm1(rng, A, 32 * A, 4, 4)
    w["policy_fc.bias"] = rng.integers(-3, 4, A).astype(np.float64)
    w["value_fc1.weight"] = _pm1(rng, 256, 32 * A, 4, 4)
    w["value_fc1.bias"] = rng.integers(-2, 3, 256).astype(np.float64)
    w["value_fc2.weight"] = rng.integers(-1, 2, (1, 256)) / 256.0
    w["value_fc2.bias"] = rng.integers(-32, 33, 1) / 256.0
    return w


def _integer(t):
    return bool((t == t.round()).all())


def reference(net64, planes):
    """float64 forward with hooks on every BatchNorm output, block output and linear layer.  -> (logits [D, A],
    pre-tanh value [D], value [D], list of violated invariants)."""
    import torch
    bad = []
    relu_in = {"bn1", "policy_bn", "value_bn"}

    def hook(name):
        def f(mod, inp, out):
            if name != "value_fc2" and not _integer(out):
                bad.append(f"{name}: not an integer")
            if out.abs().max().item() >= MAX_ACC:
                bad.append(f"{name}: accumulator >= 2^24")
            if (name.split(".")[-1] in relu_in or name.startswith("res_blocks.") and name.count(".") == 1) \
                    and out.max().item() > MAX_ACT:
                bad.append(f"{name}: ReLU output > {MAX_ACT}")
        return f

    hs = []
    for name, mod in net64.named_modules():
        if isinstance(mod, (torch.nn.BatchNorm2d, torch.nn.Linear)) or (name.startswith("res_blocks.") and name.count(".") == 1):
            hs.append(mod.register_forward_hook(hook(name)))
    feats = {}
    hs.append(net64.value_fc1.register_forward_hook(lambda mod, inp, out: feats.__setitem__("h", out)))
    hs.append(net64.value_fc2.register_forward_hook(lambda mod, inp, out: feats.__setitem__("pre", out)))
    try:
        with torch.no_grad():
            logits, value = net64(planes)
    finally:
        for h in hs:
            h.remove()
    # value_fc2 in the kernel: relu(h) * w2 per unit, summed in any order -- every partial sum must be exact
    prod = torch.relu(feats["h"]) * net64.value_fc2.weight[0]
    if not _integer(prod * 256) or (prod.abs().sum(dim=1) * 256).max().item() >= MAX_ACC:
        bad.append("value_fc2: partial sums not exact")
    return logits.cpu().numpy(), feats["pre"][:, 0].cpu().numpy(), value[:, 0].cpu().numpy(), bad


class ExactNet:
    """An integer network for (n, m, channels, blocks) that is exact on `boards`.  Attributes: state_dict (float32
    torch tensors, the reference checkpoint's keys), weights (the intended float64 integer weights), seed (the draw
    that passed), logits / pre_value / value (float64 reference on `boards`)."""

    def __init__(self, n, m, channels, blocks, seed, boards, device="cpu", tries=64):
        import torch
        from oracle import port
        self.n, self.m, self.channels, self.blocks = n, m, channels, blocks
        boards = np.asarray(boards, dtype=np.int8).reshape(-1, n, m)
        for s in range(seed, seed + tries):
            w = _draw(n, m, channels, blocks, s)
            net = port.build_net(n, m, channels, blocks)
            sd = {k: torch.tensor(w[k], dtype=v.dtype) if k in w else v for k, v in net.state_dict().items()}
            net.load_state_dict(sd)
            net64 = port.build_net(n, m, channels, blocks).double()
            net64.load_state_dict({k: torch.tensor(w[k], dtype=torch.float64) if k in w else v for k, v in net.state_dict().items()})
            net64 = net64.to(device).eval()
            planes = net64.planes(boards).double().to(device)
            logits, pre, value, bad = reference(net64, planes)
            if not bad:
                break
        else:
            raise AssertionError(f"no exact draw for {n}x{m} {channels}x{blocks} in seeds {seed}..{seed + tries - 1}: {bad}")
        self.seed, self.weights, self.state_dict = s, w, sd
        self.logits, self.pre_value, self.value = logits, pre, value


# ------------------------------------------------------------------------------------------------ packed image
def _bits(img, off, count):
    return (img[off: off + 2 * count].view(np.uint16).astype(np.uint32) << np.uint32(16)).view(np.float32).astype(np.float64)


def decode_pair_stream(img, lay, blocks):
    """The CTA-pair conv stream (the one the kernel reads): every stage [half][kc][oc/2][8] -> list over layers of
    [9 or 1 taps][N out][K in] float64."""
    off = lay["conv_stream_pair"]
    layers = []
    for l in range(2 * blocks + 2):
        stem, head = l == 0, l == 2 * blocks + 1
        taps, N, K = (1, 64, 128) if head else (9, 128, 16 if stem else 128)
        ws = []
        for _ in range(taps):
            blk = _bits(img, off, N * K).reshape(2, K // 8, N // 2, 8)       # [half][kc][oc][j]
            off += 2 * N * K
            ws.append(blk.transpose(0, 2, 1, 3).reshape(N, K))
        layers.append(np.stack(ws))
    return layers


def decode_fc_stream(img, lay, A):
    """The stage-ordered FC stream (head > K panel > M tile > stage, a stage [8 kc][rows][8]) -> (policy [A][32A],
    value_fc1 [256][32A]) float64."""
    kh, ks = 32 * A, (32 * A + 63) // 64
    n_panels = (ks + 31) // 32
    off = lay["fc_stream"]
    out = []
    for rows_total in (A, 256):
        tiles = (rows_total + 127) // 128
        wk = np.zeros((tiles * 128, ks * 64))
        for p in range(n_panels):
            for t in range(tiles):
                r = 128 if t < tiles - 1 or rows_total % 128 == 0 else (rows_total - 128 * t + 7) // 8 * 8
                for s in range(p * 32, min(ks, (p + 1) * 32)):
                    blk = _bits(img, off, 64 * r).reshape(8, r, 8)
                    off += 2 * 64 * r
                    wk[t * 128: t * 128 + r, s * 64: s * 64 + 64] = blk.transpose(1, 0, 2).reshape(r, 64)
        assert not wk[rows_total:].any() and not wk[:, kh:].any()
        out.append(wk[:rows_total, :kh])
    assert off == lay["fc_stream"] + lay["fc_stream_bytes"]
    return out


def intended_conv_layers(w, channels, blocks):
    """What the kernel should multiply with: per layer [taps][N out][K in] in the tower's padded widths (stem slots 5 / 6
    repeat the weights of the fill planes 3 / 4, for their bf16 residuals)."""
    C = channels
    stem = np.zeros((9, 128, 16))
    s = w["conv1.weight"].reshape(C, 5, 9).transpose(2, 0, 1)
    stem[:, :C, :5] = s
    stem[:, :C, 5:7] = s[:, :, 3:5]
    layers = [stem]
    for i in range(blocks):
        for conv in ("conv1", "conv2"):
            t = np.zeros((9, 128, 128))
            t[:, :C, :C] = w[f"res_blocks.{i}.{conv}.weight"].reshape(C, C, 9).transpose(2, 0, 1)
            layers.append(t)
    head = np.zeros((1, 64, 128))
    head[0, :32, :C] = w["policy_conv.weight"][:, :, 0, 0]
    head[0, 32:, :C] = w["value_conv.weight"][:, :, 0, 0]
    layers.append(head)
    return layers


def check_packed_image(net):
    """Packs net.state_dict and checks that every section the kernels or the emulation read holds the intended
    integer weights and biases exactly: both conv streams, the conv biases, the FC stream and the plain FC sections."""
    import emulate_tower as emu
    from yinyang_game_alphazero_b200 import weights
    n, m, C, blocks, w = net.n, net.m, net.channels, net.blocks, net.weights
    A = n * m
    img = weights.pack_state_dict(net.state_dict, n, m)
    lay = weights.layout(n, m, C, blocks)
    want = intended_conv_layers(w, C, blocks)
    single = emu.decode_stream(img, lay, blocks)
    pair = decode_pair_stream(img, lay, blocks)
    assert len(single) == len(pair) == len(want)
    for l, (s, p, t) in enumerate(zip(single, pair, want)):
        assert np.array_equal(np.stack([x[2] for x in s]), t), f"single-CTA conv stream, layer {l}"
        assert np.array_equal(p, t), f"CTA-pair conv stream, layer {l}"
    bias = img[lay["conv_bias"]: lay["conv_bias"] + ((2 * blocks + 1) * 128 + 64) * 4].view(np.float32).astype(np.float64)
    bns = ["bn1"] + [f"res_blocks.{i}.bn{k}" for i in range(blocks) for k in (1, 2)]
    want_b = np.concatenate([np.pad(w[b + ".bias"], (0, 128 - C)) for b in bns] + [w["policy_bn.bias"], w["value_bn.bias"]])
    assert np.array_equal(bias, want_b), "conv biases"
    wp, wv = decode_fc_stream(img, lay, A)
    assert np.array_equal(wp, w["policy_fc.weight"]) and np.array_equal(wv, w["value_fc1.weight"]), "FC stream"
    f32 = lambda off, cnt: img[off: off + 4 * cnt].view(np.float32).astype(np.float64)  # noqa: E731
    assert np.array_equal(_bits(img, lay["fc_policy_w"], lay["a_pad"] * 32 * A).reshape(-1, 32 * A)[:A], w["policy_fc.weight"])
    assert np.array_equal(_bits(img, lay["fc_value1_w"], 256 * 32 * A).reshape(256, 32 * A), w["value_fc1.weight"])
    assert np.array_equal(f32(lay["fc_policy_b"], A), w["policy_fc.bias"])
    assert np.array_equal(f32(lay["fc_value1_b"], 256), w["value_fc1.bias"])
    assert np.array_equal(f32(lay["fc_value2_w"], 256), w["value_fc2.weight"][0])
    assert np.array_equal(f32(lay["fc_value2_b"], 1), w["value_fc2.bias"])
    return img, lay


# ------------------------------------------------------------------------------------------------ positions
def positions(oracle, n, m, count, seed):
    """`count` distinct boards: the empty and the full board, random-play positions and arbitrary fills."""
    from conftest import random_play_boards
    rng = np.random.default_rng(seed)
    full = np.where(rng.random((1, n, m)) < 0.5, 1, -1).astype(np.int8)
    play, _ = random_play_boards(oracle, n, m, 3 * count, seed=seed)
    fill = rng.uniform(0, 1, (3 * count, 1, 1))
    r = rng.random((3 * count, n, m))
    arb = np.where(r < fill / 2, 1, np.where(r < fill, -1, 0)).astype(np.int8)
    seen, out = set(), []
    for b in itertools.chain([np.zeros((n, m), np.int8), full[0]], *zip(play, arb)):
        if b.tobytes() not in seen:
            seen.add(b.tobytes())
            out.append(b)
        if len(out) == count:
            break
    return np.stack(out)


def ulp_distance(a, b):
    """Distance in float32 units in the last place (same-sign finite values)."""
    ia = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    ib = np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    return np.abs(ia - ib)


def softmax64(logits):
    z = logits - logits.max(axis=1, keepdims=True)
    e = np.exp(z)
    return e / e.sum(axis=1, keepdims=True)
