"""CPU suite: bitboard packing, the product's bitboard rules header compiled for the host vs the oracle,
C-ABI surface, weight packer + emulated tower dataflow vs the fp32 network.  No compute call needs a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, golden_files, load_golden, randomise_bn
from exact_net import REPRESENTATIVES


def _host_rules(lib, bbm, boards, players, actions, n, m, flags=0, stub=False):
    bl, wh = bbm.pack_boards(boards, n, m)
    N, W = bl.shape[0], bbm.words_for(n, m)
    players = np.ascontiguousarray(players, np.int8)
    actions = np.ascontiguousarray(actions, np.int32)
    mask, nb, nw = (np.zeros((N, W), np.uint64) for _ in range(3))
    npl, ended = np.zeros(N, np.int8), np.zeros(N, np.int8)
    st = np.zeros((N, n * m + 1), np.float32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    rc = lib.yyh_rules(n, m, flags, p(bl), p(wh), p(players), p(actions), ctypes.c_long(N), p(mask), p(nb), p(nw),
                       p(npl), p(ended), p(st) if stub else None)
    assert rc == 0
    return bbm.unpack_bits(mask, n, m), bbm.unpack_boards(nb, nw, n, m), npl, ended, st


def _host_rules_sq(lib, bbm, boards, players, actions, n):
    """The line-fill rules of yy_rules_sq.cuh (square one-word boards) through the same host shim."""
    bl, wh = bbm.pack_boards(boards, n, n)
    N = bl.shape[0]
    players = np.ascontiguousarray(players, np.int8)
    actions = np.ascontiguousarray(actions, np.int32)
    mask, nb, nw = (np.zeros((N, 1), np.uint64) for _ in range(3))
    npl, ended = np.zeros(N, np.int8), np.zeros(N, np.int8)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    assert lib.yyh_rules_sq(n, p(bl), p(wh), p(players), p(actions), ctypes.c_long(N), p(mask), p(nb), p(nw), p(npl), p(ended)) == 0
    return bbm.unpack_bits(mask, n, n), bbm.unpack_boards(nb, nw, n, n), npl, ended


def _code(e):
    return np.where(e == 0.0001, 2, e).astype(np.int8)


def test_bitboard_roundtrip(yy):
    rng = np.random.default_rng(0)
    for n, m in [(4, 4), (6, 6), (8, 8), (5, 7), (16, 16), (9, 14)]:
        b = rng.integers(-1, 2, size=(37, n, m)).astype(np.int8)
        bl, wh = yy.bitboard.pack_boards(b, n, m)
        assert bl.shape == (37, yy.bitboard.words_for(n, m))
        assert np.array_equal(yy.bitboard.unpack_boards(bl, wh, n, m), b)
        a = 3 * m + 2
        assert ((int(bl[0, a >> 6]) >> (a & 63)) & 1) == int(b[0, 3, 2] == 1)   # bit a = action x*m+y


@pytest.mark.parametrize("name", golden_files("rules_"))
def test_bitboard_rules_match_reference(yy, host_rules_lib, name):
    g = load_golden(name)
    n, m, B = int(g["n"]), int(g["m"]), g["boards"]
    N = len(B)
    for pl, mk, ek in ((1, "mask_black", "ended_black"), (-1, "mask_white", "ended_white")):
        mask, _, _, ended, _ = _host_rules(host_rules_lib, yy.bitboard, B, np.full(N, pl, np.int8), g["actions"], n, m)
        assert np.array_equal(mask, g[mk]) and np.array_equal(ended, _code(g[ek]))
    _, nb, npl, _, _ = _host_rules(host_rules_lib, yy.bitboard, B, g["players"], g["actions"], n, m)
    assert np.array_equal(nb, g["next_boards"]) and np.array_equal(npl, g["next_players"])


@pytest.mark.parametrize("name", ["rules_4x4.npz", "rules_6x6.npz", "rules_8x8.npz"])
def test_line_fill_rules_match_reference(yy, host_rules_lib, name):
    """yy_rules_sq.cuh (line fills by carry propagation / Kogge-Stone, pair-based 2x2 test) against the goldens of the
    unmodified reference: masks and terminal values for both colours, next states."""
    g = load_golden(name)
    n, B = int(g["n"]), g["boards"]
    N = len(B)
    for pl, mk, ek in ((1, "mask_black", "ended_black"), (-1, "mask_white", "ended_white")):
        mask, _, _, ended = _host_rules_sq(host_rules_lib, yy.bitboard, B, np.full(N, pl, np.int8), g["actions"], n)
        assert np.array_equal(mask, g[mk]) and np.array_equal(ended, _code(g[ek]))
    _, nb, npl, _ = _host_rules_sq(host_rules_lib, yy.bitboard, B, g["players"], g["actions"], n)
    assert np.array_equal(nb, g["next_boards"]) and np.array_equal(npl, g["next_players"])


@pytest.mark.parametrize("n", [3, 4, 5, 6, 7, 8])
def test_line_fill_rules_match_step_fill_rules(yy, host_rules_lib, n):
    """Every square one-word side: the line-fill rules equal the one-cell-dilation rules of yy_rules.cuh (themselves checked
    against the oracle below) on arbitrary fills -- many components, holes, existing 2x2 blocks, full boards."""
    rng = np.random.default_rng(900 + n)
    N = 20000
    fill = rng.uniform(0, 1, size=(N, 1, 1))
    r = rng.random((N, n, n))
    B = np.where(r < fill / 2, 1, np.where(r < fill, -1, 0)).astype(np.int8)
    snake = rng.random((N // 4, n, n)) < 0.55                                  # one colour only: long thin components
    B[: N // 4] = snake.astype(np.int8)
    pl = rng.choice([1, -1], size=N).astype(np.int8)
    ac = rng.integers(-1, n * n + 1, size=N).astype(np.int32)
    a = _host_rules(host_rules_lib, yy.bitboard, B, pl, ac, n, n)[:4]
    b = _host_rules_sq(host_rules_lib, yy.bitboard, B, pl, ac, n)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


@pytest.mark.parametrize("shape", [(3, 3), (6, 6), (8, 8), (7, 9), (10, 10), (16, 16), (8, 32), (32, 8), (1, 5)])
@pytest.mark.parametrize("flags", [0, 1])
def test_bitboard_rules_match_oracle_on_arbitrary_boards(yy, host_rules_lib, oracle_mod, shape, flags):
    n, m = shape
    rng = np.random.default_rng(n * 100 + m + flags)
    N = 1500 if n * m <= 64 else 300
    fill = rng.uniform(0, 1, size=(N, 1, 1))
    r = rng.random((N, n, m))
    B = np.where(r < fill / 2, 1, np.where(r < fill, -1, 0)).astype(np.int8)
    pl = rng.choice([1, -1], size=N).astype(np.int8)
    ac = rng.integers(-1, n * m + 1, size=N).astype(np.int32)          # includes out-of-range actions
    mask, nb, npl, ended, st = _host_rules(host_rules_lib, yy.bitboard, B, pl, ac, n, m, flags, stub=True)
    ac_o = np.where(ac >= n * m, -1, ac).astype(np.int32)
    assert np.array_equal(mask, oracle_mod.legal_mask(B, pl, n, m, flags))
    onb, onp = oracle_mod.next_state(B, pl, ac_o, n, m, flags)
    assert np.array_equal(nb, onb) and np.array_equal(npl, onp)
    assert np.array_equal(ended, _code(oracle_mod.game_ended(B, pl, n, m, flags)))
    for i in range(20):
        p, v = oracle_mod.stub_predict(B[i], n, m)
        assert np.array_equal(st[i, :-1], p) and st[i, -1] == v


def test_rowcol_rule_flag(oracle_mod):
    """JS-only rule (yin_yang_game.js:338-384): completing a single-colour row is banned only with the flag."""
    b = np.zeros((1, 4, 4), np.int8)
    b[0, 0, :3] = 1
    b[0, 1, 0] = -1
    one = np.ones(1, np.int8)
    assert oracle_mod.legal_mask(b, one, 4, 4, 0)[0, 3] == 1
    assert oracle_mod.legal_mask(b, one, 4, 4, 1)[0, 3] == 0


def test_abi_exports_every_declared_symbol(yy):
    hdr = open(os.path.join(ROOT, "include", "yinyang_b200.h")).read()
    declared = set(re.findall(r"\b(yy_[a-z0-9_]+)\s*\(", hdr))
    declared |= {"yy_nn_weight_layout"}
    lib = yy._lib.lib()
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, missing
    assert set(yy._lib.SIGNATURES) >= declared - {"yy_nn_weight_layout"} | {"yy_nn_weight_layout"}
    assert lib.yy_abi_version() == 2
    assert ctypes.sizeof(yy._lib.EngineConfig) == 88


def test_no_cpu_fallback(yy):
    """Without a CUDA device every compute entry point must fail loudly (no silent CPU path)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = yy._lib.lib()
    assert lib.yy_device_count() == 0
    rc = lib.yy_legal_mask(8, 8, 0, None, None, None, None, 4, None)
    assert rc == -3 and b"no CPU fallback" in lib.yy_last_error()
    from yinyang_game_alphazero_b200 import engine
    with pytest.raises(yy.YinYangError):
        engine.Engine(rows=8, cols=8, n_games=1, n_sims=4)
    with pytest.raises(yy.YinYangError):
        engine.legal_mask_host(np.zeros((1, 8, 8), np.int8), np.ones(1, np.int8), 8, 8)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "yinyang-game-alphazero_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import oracle|from oracle)|#include\s*[\"<][^\n]*oracle|dlopen[^\n]*oracle",
                                     src, flags=re.M), f
    # developer tools and the CLI are not checkers either: only tests/, smoke() and bench.py's CPU legs run the oracle
    extra = [os.path.join(ROOT, "train_alphazero.py"), os.path.join(ROOT, "yy_b200.py")]
    extra += [os.path.join(ROOT, "tools", f) for f in os.listdir(os.path.join(ROOT, "tools")) if f.endswith(".py")]
    for path in extra:
        assert not re.search(r"^\s*(import oracle|from oracle)", open(path).read(), flags=re.M), path


@pytest.mark.parametrize("cfg", [(6, 6, 16, 2), (8, 8, 128, 1), (5, 7, 32, 1)])
def test_weight_image_and_tower_dataflow(yy, oracle_mod, cfg):
    """Packed image decoded + emulated flat-position tower (bf16 activations) vs the fp32 torch network.
    Tolerance: logits 3e-2 abs (scale ~2), value 1.5e-2 -- bf16 rounding of weights and activations."""
    import torch
    import emulate_tower as emu
    from conftest import random_play_boards
    from oracle import port
    from yinyang_game_alphazero_b200 import weights
    n, m, C, blocks = cfg
    torch.manual_seed(0)
    net = randomise_bn(port.build_net(n, m, C, blocks))
    img = weights.pack_state_dict(net.state_dict(), n, m)
    lay = weights.layout(n, m, C, blocks)
    assert img.size == lay["total"] == yy._lib.lib().yy_nn_weight_bytes(n, m, C, blocks)
    boards, _ = random_play_boards(oracle_mod, n, m, 13, seed=3)
    lg, v, _ = emu.forward(img, lay, n, m, blocks, boards)
    with torch.no_grad():
        rl, rv = net(net.planes(boards))
    np.testing.assert_allclose(lg, rl.numpy(), rtol=0, atol=3e-2)
    np.testing.assert_allclose(v, rv.numpy()[:, 0], rtol=0, atol=1.5e-2)
    assert (lg.argmax(1) == rl.numpy().argmax(1)).mean() >= 0.9


def test_bf16_rounding_helper(yy):
    import torch
    from yinyang_game_alphazero_b200 import weights
    x = np.random.default_rng(0).standard_normal(4096).astype(np.float32)
    ref = torch.from_numpy(x).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    assert np.array_equal(weights.to_bf16_bits(x), ref)


# The two reference modules a replay file meets when the reference's trainer loads it, restated: the board class the
# boards are pickled as (yin_yang_logic.py:14-22) and TrainingDataQueue.push_file (training_pipeline.py:55-73).
_REFERENCE_STAND_IN = {
    "src/__init__.py": "",
    "src/yin_yang/__init__.py": "",
    "src/yin_yang/ai/__init__.py": "",
    "src/yin_yang/yin_yang_logic.py": (
        "import numpy as np\n"
        "class YinYangLogic:\n"
        "    def __init__(self, n=8, m=8):\n"
        "        self.n, self.m = n, m\n"
        "        self.board = np.zeros((n, m), dtype=np.int8)\n"
        "    def get_board(self):\n"
        "        return self.board.copy()\n"),
    "src/yin_yang/ai/training_pipeline.py": (
        "from collections import deque\n"
        "import numpy as np\n"
        "class TrainingDataQueue:\n"
        "    def __init__(self, max_size=500000, sample_size=10000):\n"
        "        self.queue = deque(maxlen=max_size)\n"
        "    def push_file(self, file_path):\n"
        "        data = np.load(file_path, allow_pickle=True)\n"
        "        boards, policies, values = data['boards'], data['policies'], data['values']\n"
        "        for i in range(len(boards)):\n"
        "            self.queue.append((boards[i], policies[i], values[i]))\n"
        "    def __len__(self):\n"
        "        return len(self.queue)\n"),
}


def test_reference_wire_format_loads_in_the_reference(yy, tmp_path):
    """wire="reference": the .npz written by the facade must load in the reference's TrainingDataQueue
    (training_pipeline.py:55-73) in a process that cannot import this package; boards come back as the reference's
    own YinYangLogic.  The reference's source tree is used when YY_REFERENCE names it, else the restatement of its two
    modules above."""
    import subprocess
    import sys
    ref = os.environ.get("YY_REFERENCE")
    if not ref:
        ref = str(tmp_path / "reference")
        for rel, text in _REFERENCE_STAND_IN.items():
            os.makedirs(os.path.dirname(os.path.join(ref, rel)), exist_ok=True)
            with open(os.path.join(ref, rel), "w") as f:
                f.write(text)
    assert os.path.isdir(os.path.join(ref, "src", "yin_yang")), ref
    from yinyang_game_alphazero_b200 import game as game_mod, self_play
    rng = np.random.default_rng(0)
    examples = []
    for i in range(5):
        b = game_mod.YinYangLogic(6, 6)
        b.board = rng.integers(-1, 2, size=(6, 6)).astype(np.int8)
        pi = rng.random(36); pi /= pi.sum()
        examples.append((b, pi, [1, -1, 0.0001][i % 3]))
    path = str(tmp_path / "self_play_data_1.npz")
    self_play.save_examples(path, examples, 36, wire="reference")
    assert "src.yin_yang.yin_yang_logic" not in sys.modules or hasattr(sys.modules["src.yin_yang.yin_yang_logic"], "__file__")
    code = (
        "import sys, logging, numpy as np; logging.disable(logging.CRITICAL); sys.path.insert(0, %r)\n"
        "from src.yin_yang.ai.training_pipeline import TrainingDataQueue\n"
        "from src.yin_yang.yin_yang_logic import YinYangLogic\n"
        "q = TrainingDataQueue(100, 10); q.push_file(%r)\n"
        "assert len(q) == 5\n"
        "b, pi, v = q.queue[1]\n"
        "assert type(b) is YinYangLogic and b.n == 6 and b.get_board().shape == (6, 6) and pi.shape == (36,)\n"
        "assert 'yy_b200' not in sys.modules\n"
        "print('ok', int(b.get_board().sum()), float(v))\n" % (ref, path))
    r = subprocess.run([sys.executable, "-c", code], cwd=str(tmp_path), capture_output=True, text=True,
                       env={**os.environ, "PYTHONDONTWRITEBYTECODE": "1", "PYTHONPATH": ""})
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split()[0] == "ok" and int(r.stdout.split()[1]) == int(examples[1][0].board.sum())
    # native wire: this package's class
    self_play.save_examples(path, examples, 36, wire="native")
    d = np.load(path, allow_pickle=True)
    assert type(d["boards"][0]).__module__.startswith("yinyang_game_alphazero_b200")


def test_cli_imports_in_a_fresh_process(tmp_path):
    """The package's lazy attribute hook must not import modules in a cycle: run the CLI in a new interpreter up to the
    reference's "model file not found" exit (train_alphazero.py:107-109)."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "train_alphazero.py"), "--mode", "self-play", "--model-dir", str(tmp_path / "m"),
                        "--data-dir", str(tmp_path / "d")], capture_output=True, text=True, timeout=300, cwd=str(tmp_path))
    assert r.returncode == 1 and "ImportError" not in r.stderr, r.stderr[-1500:]


def test_bench_reference_arm_prints_the_contract_line(tmp_path):
    """`bench.py --impl reference` (the driver's reference arm) runs on host cores only and prints ONE JSON line with the
    same metric / unit / config keys as the B200 arm plus impl, cpu_baseline and an e2e object with zero copy bytes."""
    import json, subprocess, sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-1500:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "moves/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"].startswith("self-play moves/sec") and "configs[2]" in d["config"]["workload"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "moves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["steps"] == 1


@pytest.mark.parametrize("shape,layout,useful", [((8, 8), 3, 1.0), ((6, 6), 4, 0.84), ((16, 16), 2, 1.0), ((7, 8), 1, 0.87), ((5, 7), 0, 0.7),
                                                 ((4, 4), 0, 0.6), ((10, 10), 0, 0.75), ((12, 12), 0, 0.8), ((9, 14), 0, 0.7), ((3, 3), 0, 0.5)])
def test_tower_layouts_structural(host_tower_lib, shape, layout, useful):
    """The padded-position layouts of the tcgen05 tower (yy_tower.cuh), walked on the host: every cell of every board of a
    group is exactly one MMA row, every 3x3 tap of a cell reads the neighbouring cell of the same board or zero padding,
    nothing leaves the activation region, and in the layouts whose tiles run skewed no tap reads a cell of another tile."""
    n, m = shape
    lay, gb, T = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    u = ctypes.c_double()
    rc = host_tower_lib.yyh_tower_layout(n, m, ctypes.byref(lay), ctypes.byref(gb), ctypes.byref(T), ctypes.byref(u))
    assert rc == 0, rc
    assert lay.value == layout and u.value >= useful and gb.value * n * m <= 128 * T.value


def test_tower_layouts_structural_all_geometries(host_tower_lib):
    """The structural walk above for every board the network kernel accepts (n, m <= 32, n * m <= 256, cols + 2 <=
    TW_PAD: 500 boards); the rules' other boards are refused for being too wide."""
    lay, gb, T = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    u = ctypes.c_double()
    ok = []
    for n in range(1, 33):
        for m in range(1, 33):
            if n * m > 256:
                continue
            rc = host_tower_lib.yyh_tower_layout(n, m, ctypes.byref(lay), ctypes.byref(gb), ctypes.byref(T), ctypes.byref(u))
            if rc == -1:
                assert m + 2 > 24, (n, m)
                continue
            assert rc == 0, (n, m, rc)
            assert gb.value * n * m <= 128 * T.value, (n, m)
            ok.append((n, m))
    assert len(ok) == 500


def test_geometry_classes_have_gpu_representatives(host_tower_lib):
    """Every code-path class of the network kernel (exact_net.geometry_class) over all accepted boards has a board in
    the list the exact GPU tests run (exact_net.REPRESENTATIVES)."""
    import exact_net as X
    classes = {}
    for g in X.supported_geometries(host_tower_lib):
        classes.setdefault(X.geometry_class(X.tower_classes(host_tower_lib, *g)), []).append(g)
    covered = {X.geometry_class(X.tower_classes(host_tower_lib, n, m)) for n, m, _, _ in X.REPRESENTATIVES}
    missing = {k: v[:4] for k, v in classes.items() if k not in covered}
    assert not missing, missing
    layouts = {X.tower_classes(host_tower_lib, n, m)["layout"] for n, m, _, b in X.REPRESENTATIVES if b == 10}
    assert layouts == {k[0] for k in classes}, "a 128 x 10 net for every position layout"


@pytest.mark.parametrize("n,m,channels,blocks", REPRESENTATIVES)
def test_exact_network_packs_and_emulates_bit_exact(yy, oracle_mod, n, m, channels, blocks):
    """The integer networks of the exact GPU tests: the builder's invariants hold on the positions, the packer folds them
    into exactly the intended weights (both conv streams, biases, FC stream and sections), and for shallow nets the numpy
    emulation of the kernel's dataflow reproduces the float64 reference's logits bit for bit."""
    import emulate_tower as emu
    import exact_net as X
    boards = X.positions(oracle_mod, n, m, 12, seed=n * 100 + m)
    net = X.ExactNet(n, m, channels, blocks, seed=1000 + n * 100 + m, boards=boards)
    assert np.array_equal(net.logits, np.round(net.logits)) and np.all(np.abs(net.logits) < 2 ** 24)
    img, lay = X.check_packed_image(net)
    if blocks <= 2:
        lg, v, _ = emu.forward(img, lay, n, m, blocks, boards)
        assert np.array_equal(lg, net.logits.astype(np.float32))
        assert X.ulp_distance(v, np.tanh(net.pre_value).astype(np.float32)).max() <= 2
