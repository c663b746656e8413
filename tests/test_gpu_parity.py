"""GPU parity tests (run on the B200 box with -m gpu).  Every check calls the CUDA path through the C ABI
(ctypes) and compares with the oracle / the golden fixtures.  Integer work is bit-exact; the bf16 network is
checked against the fp32 torch restatement at the stated tolerance and against the numpy emulation of the
kernel's own dataflow at a much tighter one."""
import numpy as np
import pytest

from conftest import golden_files, load_golden, random_play_boards, randomise_bn
from exact_net import REPRESENTATIVES

pytestmark = pytest.mark.gpu


def _code(e):
    return np.where(e == 0.0001, 2, e).astype(np.int8)


@pytest.fixture(scope="module")
def eng(yy):
    from yinyang_game_alphazero_b200 import engine
    return engine


# ------------------------------------------------------------------------------------------------ tcgen05 probe
@pytest.mark.parametrize("N,K,off", [(128, 64, 0), (128, 128, 0), (64, 64, 0), (128, 64, 8), (128, 64, 1),
                                      (128, 64, 9), (128, 64, 23), (256, 32, 5), (16, 16, 3)])
def test_umma_descriptor_probe(yy, N, K, off):
    """C = A[off:off+128] @ B^T on tcgen05 with the tower kernel's no-swizzle K-major descriptors, including
    start addresses that are NOT multiples of 8 rows (what a 3x3 tap shift produces)."""
    import ctypes
    import torch
    rows = 160
    g = torch.Generator(device="cpu").manual_seed(N * 1000 + K + off)
    A = (torch.randn(rows, K, generator=g)).to(torch.bfloat16).cuda()
    B = (torch.randn(N, K, generator=g)).to(torch.bfloat16).cuda()
    C = torch.zeros(128, N, dtype=torch.float32, device="cuda")
    lib = yy._lib.lib()
    rc = lib.yy_probe_umma(ctypes.c_void_p(A.data_ptr()), ctypes.c_void_p(B.data_ptr()), ctypes.c_void_p(C.data_ptr()),
                           rows, N, K, off, 0, None)
    assert rc == 0, lib.yy_last_error()
    torch.cuda.synchronize()
    ref = A[off:off + 128].float() @ B.float().t()
    err = (C - ref).abs().max().item()
    assert err < 1e-3 * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("grp,off", [(9, 0), (9, 10), (9, 19), (10, 3), (17, 1)])
def test_umma_strided_row_groups(yy, grp, off):
    """SBO != 128: the MMA's 8-row groups start every `grp` rows (SBO = grp*16 B), so C row m reads A row
    off + (m/8)*grp + m%8 -- the row-aligned tower layout (one board row per group, zero column skipped)."""
    import ctypes
    import torch
    N, K = 128, 64
    rows = off + 15 * grp + 8 + 3
    g = torch.Generator(device="cpu").manual_seed(grp * 100 + off)
    A = torch.randn(rows, K, generator=g).to(torch.bfloat16).cuda()
    B = torch.randn(N, K, generator=g).to(torch.bfloat16).cuda()
    C = torch.zeros(128, N, dtype=torch.float32, device="cuda")
    lib = yy._lib.lib()
    rc = lib.yy_probe_umma(ctypes.c_void_p(A.data_ptr()), ctypes.c_void_p(B.data_ptr()), ctypes.c_void_p(C.data_ptr()),
                           rows, N, K, off, grp, None)
    assert rc == 0, lib.yy_last_error()
    torch.cuda.synchronize()
    idx = torch.tensor([off + (m // 8) * grp + m % 8 for m in range(128)], device="cuda")
    ref = A[idx].float() @ B.float().t()
    assert (C - ref).abs().max().item() < 1e-3 * max(1.0, ref.abs().max().item())


# ------------------------------------------------------------------------------------------------ rules
@pytest.mark.parametrize("name", golden_files("rules_"))
def test_rules_match_reference_golden(eng, name):
    g = load_golden(name)
    n, m, B = int(g["n"]), int(g["m"]), g["boards"]
    N = len(B)
    one = np.ones(N, np.int8)
    assert np.array_equal(eng.legal_mask_host(B, one, n, m), g["mask_black"])
    assert np.array_equal(eng.legal_mask_host(B, -one, n, m), g["mask_white"])
    nb, npl = eng.next_state_host(B, g["players"], g["actions"], n, m)
    assert np.array_equal(nb, g["next_boards"]) and np.array_equal(npl, g["next_players"])
    assert np.array_equal(eng.ended_host(B, one, n, m), g["ended_black"])
    assert np.array_equal(eng.ended_host(B, -one, n, m), g["ended_white"])


@pytest.mark.parametrize("name", golden_files("rowcol_"))
def test_rowcol_rule_matches_js_transcription_golden(eng, name):
    """YY_RULE_ROWCOL on the GPU against the literal transcription of the browser game's rule (yin_yang_game.js:186-232,
    :338-384; tests/golden/make_golden_rowcol.py), both colours, incl. boards with complete and nearly complete lines."""
    g = load_golden(name)
    n, m, B = int(g["n"]), int(g["m"]), g["boards"]
    one = np.ones(len(B), np.int8)
    assert np.array_equal(eng.legal_mask_host(B, one, n, m, eng.RULE_ROWCOL), g["mask_black"])
    assert np.array_equal(eng.legal_mask_host(B, -one, n, m, eng.RULE_ROWCOL), g["mask_white"])


def test_env_step_packed_host_buffers(eng, oracle_mod):
    """env_step_host_packed: packed uint64 boards in host memory in and out (the C ABI's own layout)."""
    from yinyang_game_alphazero_b200 import bitboard
    n = m = 8
    boards, players = random_play_boards(oracle_mod, n, m, 3000, seed=77)
    rng = np.random.default_rng(5)
    masks_o = oracle_mod.legal_mask(boards, players, n, m)
    actions = np.array([rng.choice(np.flatnonzero(mk)) if mk.any() else -1 for mk in masks_o], dtype=np.int32)
    mo, bo, po, ro = oracle_mod.env_step(boards, players, actions, n, m)
    bk, wh = bitboard.pack_boards(boards, n, m)
    hm, hb, hw, hp, hr = eng.env_step_host_packed(bk, wh, players, actions, n, m)
    assert np.array_equal(bitboard.unpack_bits(hm, n, m), mo) and np.array_equal(bitboard.unpack_boards(hb, hw, n, m), bo)
    assert np.array_equal(hp, po) and np.array_equal(eng.result_from_code(hr), ro)


@pytest.mark.parametrize("shape,flags", [((8, 8), 0), ((8, 8), 1), ((6, 6), 0), ((16, 16), 0), ((10, 10), 1), ((5, 7), 0)])
def test_env_step_matches_oracle(eng, oracle_mod, shape, flags):
    n, m = shape
    N = 4096 if n * m <= 64 else 512
    rng = np.random.default_rng(7 + n)
    boards, players = random_play_boards(oracle_mod, n, m, N, seed=11 + n)
    arb = rng.random((N // 4, n, m))
    boards[: N // 4] = np.where(arb < 0.2, 1, np.where(arb < 0.4, -1, 0))        # arbitrary (non-legal-play) boards too
    masks_o = oracle_mod.legal_mask(boards, players, n, m, flags)
    actions = np.array([rng.choice(np.flatnonzero(mk)) if mk.any() and rng.random() < 0.8 else rng.integers(-1, n * m)
                        for mk in masks_o], dtype=np.int32)
    mo, bo, po, ro = oracle_mod.env_step(boards, players, actions, n, m, flags)
    mg, bg, pg, rg = eng.env_step_host(boards, players, actions, n, m, flags)
    assert np.array_equal(mg, mo) and np.array_equal(bg, bo) and np.array_equal(pg, po) and np.array_equal(rg, ro)


def test_env_step_full_config2(eng, oracle_mod):
    """BASELINE.json configs[1]: 65,536 synthetic random-play 8x8 boards (device generator), whole set checked
    bit-exact against the C oracle; plus empty and ragged (count = 1, 0) batches."""
    import torch
    n = m = 8
    N = 65536
    plies = torch.arange(N, dtype=torch.int32) % 52
    black, white, players = eng.random_playout(N, plies, n, m, seed=0xC0FFEE)
    bl, wh = black.cpu().numpy().view(np.uint64), white.cpu().numpy().view(np.uint64)
    from yinyang_game_alphazero_b200 import bitboard
    boards = bitboard.unpack_boards(bl, wh, n, m)
    pl = players.cpu().numpy()
    stones = np.abs(boards).sum(axis=(1, 2))
    assert stones.max() <= 51 and stones.mean() > 15                      # really are mid-game positions
    assert np.all((boards == 1).sum(axis=(1, 2)) >= (boards == -1).sum(axis=(1, 2)) - 26)
    masks_o = oracle_mod.legal_mask(boards, pl, n, m)
    rng = np.random.default_rng(0)
    actions = np.array([rng.choice(np.flatnonzero(mk)) if mk.any() else -1 for mk in masks_o], dtype=np.int32)
    mo, bo, po, ro = oracle_mod.env_step(boards, pl, actions, n, m)
    act_d = torch.from_numpy(actions).cuda()
    mask_d, res_d = eng.env_step(black, white, players, act_d, n, m)
    assert np.array_equal(bitboard.unpack_bits(mask_d.cpu().numpy().view(np.uint64), n, m), mo)
    assert np.array_equal(bitboard.unpack_boards(black.cpu().numpy().view(np.uint64), white.cpu().numpy().view(np.uint64), n, m), bo)
    assert np.array_equal(players.cpu().numpy(), po)
    assert np.array_equal(eng.result_from_code(res_d.cpu().numpy()), ro)
    for cnt in (0, 1):
        out = eng.env_step_host(boards[:cnt], pl[:cnt], actions[:cnt], n, m)
        assert out[0].shape[0] == cnt


# ------------------------------------------------------------------------------------------------ MCTS (deterministic-prior mode)
@pytest.mark.parametrize("name", golden_files("mcts_"))
def test_mcts_visit_counts_match_reference_golden(eng, name):
    g = load_golden(name)
    n, m = int(g["n"]), int(g["m"])
    e = eng.Engine(rows=n, cols=m, n_games=1, n_sims=int(g["sims"]), evaluator="stub", cpuct=float(g["cpuct"]))
    noise = [g["noise"]] if g["noise"].size else None
    counts, cw = e.search_host(g["board"][None], np.array([int(g["player"])], np.int8), noise=noise)
    assert np.array_equal(counts[0], g["counts"])
    assert np.array_equal(cw[0], g["child_w"])                            # float32 value sums, bit for bit
    e.close()


@pytest.mark.parametrize("step_kernels", [False, True])
@pytest.mark.parametrize("shape,sims,games", [((8, 8), 200, 96), ((6, 6), 150, 64), ((4, 4), 300, 64), ((16, 16), 40, 8),
                                              ((8, 8), 60, 700), ((8, 8), 800, 40), ((16, 16), 1600, 6), ((6, 6), 100, 48)])
def test_mcts_matches_oracle_many_games(eng, oracle_mod, shape, sims, games, step_kernels):
    """Both search drivers -- ONE persistent kernel per search (default, csrc/yy_fused.cu) and one tree-step launch
    per simulation (YY_MODE_STEP_KERNELS) -- must reproduce the oracle bit for bit.  700 games: several games per
    CTA and more than one heads batch per CTA in the persistent kernel.  8x8 / 800, 16x16 / 1,600 and 6x6 / 100 are the
    simulation budgets BASELINE.json's configs state, on early, middle and late random-play positions."""
    n, m = shape
    boards, players = random_play_boards(oracle_mod, n, m, games, seed=5 + n)
    rng = np.random.default_rng(1)
    noise = []
    for i in range(games):
        k = int(oracle_mod.legal_mask(boards[i][None], players[i:i + 1], n, m).sum())
        noise.append(rng.dirichlet([0.3] * k) if (i % 3 == 0 and k > 0) else None)
    e = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="stub", cpuct=1.25, step_kernels=step_kernels)
    counts, cw = e.search_host(boards, players, noise=noise)
    for i in range(0, games, 1 if games <= 100 else 7):
        r = oracle_mod.mcts_search(boards[i], int(players[i]), n, m, sims, cpuct=1.25, noise=noise[i])
        assert np.array_equal(counts[i], r["counts"]), i
        assert np.array_equal(cw[i], r["child_w"]), i
    e.close()


@pytest.mark.parametrize("K", [4, 16])
def test_mcts_virtual_loss_throughput_mode(eng, oracle_mod, K):
    """leaves_per_step = K > 1: K in-flight simulations per game per step with virtual loss.  Not bit-exact by
    design; invariants: every simulation is accounted for (root child visits sum to n_sims), value sums stay
    bounded, the arena does not overflow, and the search still concentrates on the deterministic search's
    preferred moves (the 3 most visited actions overlap)."""
    n = m = 8
    games, sims = 32, 256
    boards, players = random_play_boards(oracle_mod, n, m, games, seed=21, max_frac=0.5)
    e1 = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="stub")
    c1, _ = e1.search_host(boards, players)
    e1.close()
    ek = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="stub", leaves_per_step=K)
    ck, wk = ek.search_host(boards, players)
    st = ek.stats()
    ek.close()
    assert st.overflow == 0
    has_moves = c1.sum(axis=1) > 0
    assert np.array_equal(ck.sum(axis=1)[has_moves], np.full(has_moves.sum(), sims))
    assert np.all(np.abs(wk) <= ck + 1e-3)                      # |W| <= N: every virtual loss was taken back
    agree = [len(set(np.argsort(-c1[i])[:3]) & set(np.argsort(-ck[i])[:3])) for i in np.flatnonzero(has_moves)]
    assert np.mean(agree) >= 1.5


def test_mcts_external_evaluator_seam(eng, oracle_mod):
    """The duck-typed predict seam: priors/values supplied by the caller each step (here: the oracle's stub,
    computed on the host) must give the same visit counts as the fused stub evaluator."""
    import torch
    from yinyang_game_alphazero_b200 import bitboard
    n = m = 6
    games, sims = 8, 60
    boards, players = random_play_boards(oracle_mod, n, m, games, seed=2)
    e = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="external")
    b, w = bitboard.pack_boards(boards, n, m)
    bd, wd = torch.from_numpy(b.view(np.int64)).cuda(), torch.from_numpy(w.view(np.int64)).cuda()
    e.search_begin(bd, wd, torch.from_numpy(players).cuda())
    active = games
    steps = 0
    while active:
        lb, lw, act = e.leaf_batch()
        leaf = bitboard.unpack_boards(lb.cpu().numpy().view(np.uint64), lw.cpu().numpy().view(np.uint64), n, m)
        pr = np.zeros((games, n * m), np.float32); va = np.zeros(games, np.float32)
        for i in range(games):
            pr[i], va[i] = oracle_mod.stub_predict(leaf[i], n, m)
        active = e.search_advance(torch.from_numpy(pr).cuda(), torch.from_numpy(va).cuda())
        steps += 1
        assert steps <= sims + 2
    counts, _ = e.search_counts()
    for i in range(games):
        r = oracle_mod.mcts_search(boards[i], int(players[i]), n, m, sims)
        assert np.array_equal(counts[i].cpu().numpy(), r["counts"])
    e.close()


# ------------------------------------------------------------------------------------------------ network
@pytest.mark.parametrize("cfg", [(8, 8, 128, 10, 300, False), (8, 8, 128, 10, 64, True), (8, 8, 128, 0, 40, True),
                                 (8, 8, 128, 1, 40, True), (6, 6, 128, 3, 64, True), (8, 8, 32, 2, 50, True),
                                 (16, 16, 128, 1, 9, True), (5, 7, 64, 2, 33, True), (8, 8, 128, 1, 37, True),
                                 (16, 16, 64, 2, 35, False), (8, 8, 128, 2, 1000, False), (6, 6, 128, 1, 5000, True)]
                         # one board of every geometry class of the kernel (tests/exact_net.py REPRESENTATIVES)
                         + [(n, m, C, min(b, 2), 40, True) for n, m, C, b in REPRESENTATIVES if (n, m) not in {(8, 8), (6, 6), (16, 16), (5, 7)}])
def test_network_matches_fp32_reference(eng, oracle_mod, cfg):
    """bf16 tcgen05 tower + heads vs the fp32 torch network (reference semantics, neural_network.py:94-154).
    Stated tolerance (bf16 weights + bf16 inter-layer activations, fp32 accumulate), measured headroom ~2x:
        logits  max|err| <= 0.015 * max|logit| + 0.01      value  max|err| <= 0.06
        policy  total-variation distance <= 0.05           top-1 agreement >= 80 %
    cfg[-1] False = reference initialisation (xavier weights, identity BN), True = random BN statistics.
    Shallow nets (<= 1 block) are also compared with the numpy emulation of the kernel's own dataflow from the
    same packed image at 2e-3: there only the fp32 summation order differs, so this pins the kernel logic."""
    import torch
    import emulate_tower as emu
    from oracle import port
    from yinyang_game_alphazero_b200 import weights
    n, m, C, blocks, count, rnd = cfg
    torch.manual_seed(0)
    net = port.build_net(n, m, C, blocks)
    net = randomise_bn(net) if rnd else net.eval()
    e = eng.Engine(rows=n, cols=m, n_games=max(count, 4), n_sims=1, evaluator="nn", state_dict=net.state_dict())
    boards, _ = random_play_boards(oracle_mod, n, m, count, seed=9)
    policy, value, logits = e.evaluate_host(boards, want_logits=True)
    with torch.no_grad():
        rl, rv = net(net.planes(boards))
        rp = torch.softmax(rl, dim=1).numpy()
    rl, rv = rl.numpy(), rv.numpy()[:, 0]
    if blocks <= 1:
        img = weights.pack_state_dict(net.state_dict(), n, m)
        lay = weights.layout(n, m, C, blocks)
        k = min(count, 24)
        el, ev, _ = emu.forward(img, lay, n, m, blocks, boards[:k])
        np.testing.assert_allclose(logits[:k], el, rtol=0, atol=2e-3)
        np.testing.assert_allclose(value[:k], ev, rtol=0, atol=2e-3)
    np.testing.assert_allclose(logits, rl, rtol=0, atol=0.015 * float(np.abs(rl).max()) + 0.01)
    np.testing.assert_allclose(value, rv, rtol=0, atol=0.06)
    np.testing.assert_allclose(policy.sum(axis=1), 1.0, atol=1e-5)
    assert 0.5 * np.abs(policy - rp).sum(axis=1).max() <= 0.05
    assert (logits.argmax(1) == rl.argmax(1)).mean() >= 0.8
    # a second call on the same inputs is bit-identical (fixed summation order, no atomics)
    p2, v2, l2 = e.evaluate_host(boards, want_logits=True)
    assert np.array_equal(l2, logits) and np.array_equal(v2, value)
    e.close()


@pytest.mark.parametrize("n,count", [(8, 500), (6, 700), (16, 40)])
def test_tower_tile_skew_is_bit_identical_to_lockstep(eng, oracle_mod, n, count):
    """The tile skew of the persistent kernel (the MMA issuer walks the first and last stages of a layer tile by tile,
    per-tile barriers) only reorders WHEN a tile's MMAs and epilogue run, never the order of a tile's own accumulation:
    logits, policy and value must equal, bit for bit, those of the lock-step walk (developer flag bit 1) and of the
    half-group ping-pong (bit 0) -- full groups, a partial last group and several heads batches per CTA included."""
    import torch
    from oracle import port
    torch.manual_seed(1)
    net = randomise_bn(port.build_net(n, n, 128, 2))
    boards, _ = random_play_boards(oracle_mod, n, n, count, seed=21)
    e = eng.Engine(rows=n, cols=n, n_games=count, n_sims=1, evaluator="nn", state_dict=net.state_dict())
    outs = []
    for flags in (0, 2, 1):
        e.L.yy_engine_set_debug_flags(e.handle, flags)
        outs.append(e.evaluate_host(boards, want_logits=True))
    e.L.yy_engine_set_debug_flags(e.handle, 0)
    e.close()
    for other in outs[1:]:
        for a, b in zip(outs[0], other):
            assert np.array_equal(a, b)


def test_network_search_persistent_vs_step_kernels(eng, oracle_mod):
    """Network-driven search: ONE persistent launch per search (tower + FC heads + tree step fused) against one
    network launch + one tree-step launch per simulation (YY_MODE_STEP_KERNELS).  Same network code, same tree code:
    the visit counts must be identical."""
    import torch
    from oracle import port
    n = m = 8
    games, sims = 300, 48
    torch.manual_seed(3)
    net = randomise_bn(port.build_net(n, m, 128, 2))
    boards, players = random_play_boards(oracle_mod, n, m, games, seed=77, max_frac=0.6)
    res = []
    for sk in (False, True):
        e = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="nn", state_dict=net.state_dict(), step_kernels=sk)
        c, w = e.search_host(boards, players)
        st = e.stats()
        assert st.overflow == 0
        res.append((c, w))
        pol, val = e.evaluate_host(boards)[:2]
        res.append((pol, val))
        e.close()
    (c0, w0), (p0, v0), (c1, w1), (p1, v1) = res
    assert np.array_equal(p0, p1) and np.array_equal(v0, v1)
    has_moves = c1.sum(axis=1) > 0
    assert np.array_equal(c0.sum(axis=1), c1.sum(axis=1))
    assert np.all(c0.sum(axis=1)[has_moves] == sims)
    assert np.array_equal(c0, c1) and np.array_equal(w0, w1)


@pytest.mark.parametrize("n,sims", [(8, 800), (16, 1600), (6, 100)])
def test_search_full_config_replica_properties(eng, oracle_mod, n, sims):
    """BASELINE.json configs[2] at full size (8x8, 800 simulations, 4,096 concurrent games, 128x10 network), configs[4]'s
    per-GPU share (16x16, 1,600 simulations, 4,096 of the 32,768 games) and configs[0]'s board and budget (6x6, 100
    simulations) at 4,096 games, through
    size-independent properties: 64 distinct positions are each given to 64 of the 4,096 slots in a shuffled order.
    (1) every replica of a position returns the same visit counts and child value sums bit for bit, whichever slot /
    CTA pair / SM searched it; (2) the same 64 positions searched by a 64-game engine give those counts too (batch-size
    independence); (3) every search with a legal move spends exactly 800 simulations on legal actions only."""
    import torch
    from oracle import port
    m = n
    games, distinct = 4096, 64
    torch.manual_seed(5)
    net = randomise_bn(port.build_net(n, m, 128, 10))
    base_b, base_p = random_play_boards(oracle_mod, n, m, distinct, seed=123, max_frac=0.7)
    base_b[0] = 0; base_p[0] = 1                                  # the empty board (the benchmark's root) is one of them
    slot_pos = np.random.default_rng(9).permutation(np.repeat(np.arange(distinct), games // distinct))
    e = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="nn", state_dict=net.state_dict())
    counts, cw = e.search_host(base_b[slot_pos], base_p[slot_pos])
    st = e.stats()
    e.close()
    assert st.overflow == 0
    legal = oracle_mod.legal_mask(base_b, base_p, n, m).astype(bool)
    for k in range(distinct):
        rep = np.flatnonzero(slot_pos == k)
        assert np.all(counts[rep] == counts[rep[0]]), f"position {k}: replicas disagree on visit counts"
        assert np.all(cw[rep] == cw[rep[0]]), f"position {k}: replicas disagree on value sums"
        c = counts[rep[0]]
        assert c.sum() == (sims if legal[k].any() else 0) and not c[~legal[k]].any()
    small = eng.Engine(rows=n, cols=m, n_games=distinct, n_sims=sims, evaluator="nn", state_dict=net.state_dict())
    c2, w2 = small.search_host(base_b, base_p)
    small.close()
    first = np.array([np.flatnonzero(slot_pos == k)[0] for k in range(distinct)])
    assert np.array_equal(c2, counts[first]) and np.array_equal(w2, cw[first])


# ------------------------------------------------------------------------------------------------ dataset / augmentation
@pytest.mark.parametrize("name", golden_files("augment_"))
def test_augmentation_matches_reference_golden(eng, name):
    """yy_augment_samples vs create_dataset_from_games of the unmodified reference (data_utils.py:182-215): float32
    planes, policies and values of all 8 forms, bit for bit; both policy sources (visit counts / float32 policy)."""
    g = load_golden(name)
    n, m = int(g["n"]), int(g["m"])
    planes, pol, vals = eng.augment_samples_host(g["boards"], n, m, counts=g["counts"], values=g["values"])
    assert np.array_equal(planes, g["planes"]) and np.array_equal(pol, g["policies"]) and np.array_equal(vals, g["out_values"])
    planes2, pol2, _ = eng.augment_samples_host(g["boards"], n, m, policy=g["policies"][0::8])
    assert np.array_equal(planes2, g["planes"]) and np.array_equal(pol2, g["policies"])


@pytest.mark.parametrize("shape,count", [((8, 8), 5000), ((6, 6), 777), ((16, 16), 300), ((3, 3), 33), ((8, 8), 0)])
def test_augmentation_matches_oracle(eng, oracle_mod, shape, count):
    n, m = shape
    rng = np.random.default_rng(n * 100 + count)
    boards = rng.integers(-1, 2, size=(count, n, m)).astype(np.int8)
    counts = (rng.integers(0, 65535, size=(count, n * m)) * (rng.random((count, n * m)) < 0.5)).astype(np.uint16)
    if count:
        counts[::11] = 0
    values = rng.choice([1.0, -1.0, 0.0001], size=count)
    planes, pol, vals = eng.augment_samples_host(boards, n, m, counts=counts, values=values)
    rp, rq, rv = oracle_mod.augment_dataset(boards, counts, values, n, m)
    assert planes.shape == rp.shape and np.array_equal(planes, rp)
    assert np.array_equal(pol, rq) and np.array_equal(vals, rv)
    # size-independent properties: every form is a permutation of the identity form; policies still sum to one
    if count:
        assert np.array_equal(np.sort(pol.reshape(count, 8, -1), axis=2), np.sort(pol.reshape(count, 8, -1)[:, :1], axis=2).repeat(8, 1))
        np.testing.assert_allclose(pol.sum(axis=1), 1.0, atol=1e-5)


def test_augmentation_into_caller_buffers(eng, oracle_mod):
    """out= : the second call writes into the first call's tensors (caller-allocated outputs, as over the C ABI)."""
    import torch
    n = 8
    rng = np.random.default_rng(4)
    b1, p1 = random_play_boards(oracle_mod, n, n, 300, seed=31)
    b2, p2 = random_play_boards(oracle_mod, n, n, 300, seed=32)
    c1 = rng.integers(0, 800, size=(300, n * n)).astype(np.uint16); c2 = rng.integers(0, 800, size=(300, n * n)).astype(np.uint16)
    v = torch.ones(300, device="cuda")
    dev = lambda boards: eng.pack_boards_dev(boards, n, n)
    cnt = lambda c: torch.from_numpy(c.view(np.int16)).cuda()
    out = eng.augment_samples(*dev(b1), n, n, counts=cnt(c1), values=v)
    ptrs = [t.data_ptr() for t in out]
    out2 = eng.augment_samples(*dev(b2), n, n, counts=cnt(c2), values=v, out=out)
    assert [t.data_ptr() for t in out2] == ptrs
    rp, rq, rv = oracle_mod.augment_dataset(b2, c2, np.ones(300), n, n)
    assert np.array_equal(out2[0].cpu().numpy(), rp) and np.array_equal(out2[1].cpu().numpy(), rq) and np.array_equal(out2[2].cpu().numpy(), rv)


@pytest.mark.parametrize("shape", [(5, 7), (8, 8), (3, 9)])
def test_dataset_without_augmentation_any_shape(eng, oracle_mod, shape):
    """yy_dataset_samples (create_dataset_from_games(..., augment=False), DataProcessor.preprocess_sample): planes and
    policies of every record, identity form only -- also on the non-square boards the rotations exclude."""
    n, m = shape
    rng = np.random.default_rng(n * 10 + m)
    boards = rng.integers(-1, 2, size=(200, n, m)).astype(np.int8)
    counts = rng.integers(0, 500, size=(200, n * m)).astype(np.uint16)
    counts[::9] = 0
    values = rng.choice([1.0, -1.0, 0.0001], size=200)
    planes, pol, vals = eng.augment_samples_host(boards, n, m, counts=counts, values=values, forms=1)
    ref = oracle_mod.input_planes(boards, n, m)
    tot = counts.sum(axis=1, keepdims=True).astype(np.float64)
    rpol = np.where(tot > 0, counts / np.maximum(tot, 1.0), 1.0 / (n * m)).astype(np.float32)
    assert planes.shape == (200, 5, n, m) and np.array_equal(planes, ref)
    assert np.array_equal(pol, rpol) and np.array_equal(vals, values.astype(np.float32))


def test_augmentation_rejects_non_square(eng):
    from yinyang_game_alphazero_b200 import YinYangError
    with pytest.raises(YinYangError):
        eng.augment_samples_host(np.zeros((2, 5, 7), np.int8), 5, 7, counts=np.ones((2, 35), np.uint16))


# ------------------------------------------------------------------------------------------------ self-play driver
def test_selfplay_records_match_oracle_search(eng, oracle_mod):
    """Every replay record's visit counts must equal the oracle's search from that record's board (noise off,
    stub evaluator), games must progress by legal single-stone moves, results must be terminal codes."""
    n = m = 6
    games, sims, moves = 24, 40, 30
    e = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="stub", dirichlet_epsilon=0.0, seed=123,
                   search_as_black=False)
    e.selfplay_run(moves)
    st = e.stats()
    assert st.moves == games * moves and st.examples == games * moves and st.overflow == 0
    rp = e.replay()
    assert rp["boards"].shape[0] == games * moves
    for i in range(0, games * moves, 3):
        r = oracle_mod.mcts_search(rp["boards"][i], int(rp["player"][i]), n, m, sims)
        assert np.array_equal(rp["counts"][i].astype(np.int32), r["counts"]), i
    # per-game trajectories: consecutive plies add exactly one stone of the mover's colour
    order = np.lexsort((rp["ply"], rp["game_serial"]))
    for a, b in zip(order[:-1], order[1:]):
        if rp["game_serial"][a] == rp["game_serial"][b] and rp["ply"][b] == rp["ply"][a] + 1:
            diff = rp["boards"][b].astype(int) - rp["boards"][a].astype(int)
            assert np.abs(diff).sum() == 1 and diff.sum() == rp["player"][a]
    assert st.games_finished > 0
    z = rp["z"][rp["finished"]]
    assert np.all(np.isin(z, [1.0, -1.0, 0.0001]))
    fin = np.unique(rp["game_serial"][rp["finished"]])
    assert len(fin) >= st.games_finished - games
    e.close()


def test_selfplay_reference_player_semantics(eng, oracle_mod):
    """SURVEY Q5 (self_play.py:99,135-137,163): default mode searches every position as player 1 and applies
    the chosen action with the real player -- an action illegal for the real player is silently dropped."""
    n = m = 6
    games, sims, moves = 16, 24, 12
    e = eng.Engine(rows=n, cols=m, n_games=games, n_sims=sims, evaluator="stub", dirichlet_epsilon=0.0, seed=5)
    e.selfplay_run(moves)
    rp = e.replay()
    for i in range(0, games * moves, 5):
        r = oracle_mod.mcts_search(rp["boards"][i], 1, n, m, sims)       # searched as black whatever the mover
        assert np.array_equal(rp["counts"][i].astype(np.int32), r["counts"]), i
    e.close()


def _engine_games(e, total, chunk=4000):
    """Runs rolling self-play until `total` games (the quota) are finished; returns {serial: (boards, pi, z)}."""
    e.selfplay_set_quota(total)
    for _ in range(2000):
        e.selfplay_advance(chunk)
        if e.stats().games_finished >= total:
            break
    st = e.stats()
    assert st.games_finished == total and st.overflow == 0 and st.examples <= e.replay_capacity
    rp = e.replay()
    out = {}
    order = np.lexsort((rp["ply"], rp["game_serial"]))
    for s in range(total):
        idx = order[rp["game_serial"][order] == s]
        assert np.array_equal(rp["ply"][idx], np.arange(len(idx))) and rp["finished"][idx].all()
        out[s] = (rp["boards"][idx], rp["pi"][idx], rp["z"][idx])
    return out


@pytest.mark.parametrize("name", golden_files("selfplay_"))
def test_selfplay_episode_matches_reference_golden(eng, name):
    """SURVEY 8a-15: a whole game played by the engine's episode driver (prepare / noise / search / move inside the
    persistent kernel) against the same game played by the UNMODIFIED SelfPlayWorker.play_game on the same recorded
    random stream (tests/golden/make_golden_selfplay.py): every stored position, pi in float64, and z -- including the
    pass / double-pass branch (1e-4 for every example), decisive results (+1 / -1 for every example: the double sign
    flip of self_play.py:172-181), moves silently dropped for the real player, and the argmax branch after the
    temperature threshold."""
    g = load_golden(name)
    n, m, A = int(g["n"]), int(g["m"]), int(g["n"]) * int(g["m"])
    noise = np.zeros((1, A)); noise[0, :g["noise"].size] = g["noise"]
    e = eng.Engine(rows=n, cols=m, n_games=1, n_sims=int(g["sims"]), evaluator="stub", cpuct=float(g["cpuct"]),
                   dirichlet_epsilon=float(g["eps"]), dirichlet_alpha=float(g["alpha"]),
                   temperature_threshold=int(g["temperature_threshold"]), replay_capacity=4 * A + 64)
    e.selfplay_set_random_stream(g["uniforms"][None], noise)
    boards, pi, z = _engine_games(e, 1)[0]
    e.close()
    assert np.array_equal(boards, g["boards"])
    assert np.array_equal(pi, g["pis"])                       # float64, bit for bit
    assert np.array_equal(z, g["zs"])


@pytest.mark.parametrize("n,m,sims,tt,sab", [(4, 4, 50, 3, True), (6, 6, 40, 8, True), (5, 7, 30, 10, True), (8, 8, 24, 10, True),
                                             (6, 6, 40, 8, False)])
def test_selfplay_episodes_match_oracle(eng, oracle_mod, n, m, sims, tt, sab):
    """48 whole games on 16 slots (three generations per slot, rolling) against the oracle's play_game on the same
    recorded stream -- game s is the same game whichever slot played it.  Also the side-to-move search mode."""
    A, total, P = n * m, 48, 4 * n * m
    rng = np.random.default_rng(n * 100 + m)
    uniforms = rng.random((total, P))
    noise = np.stack([rng.dirichlet([0.3] * A) for _ in range(total)])
    e = eng.Engine(rows=n, cols=m, n_games=16, n_sims=sims, evaluator="stub", temperature_threshold=tt, search_as_black=sab,
                   replay_capacity=total * P)
    e.selfplay_set_random_stream(uniforms, noise)
    games = _engine_games(e, total, chunk=701)
    e.close()
    kinds = set()
    for s in range(total):
        b, pi, z, kind = oracle_mod.play_game(n, m, sims, uniforms[s], noise[s], temperature_threshold=tt, search_as_black=sab)
        kinds.add((kind, float(z[0])))
        assert np.array_equal(games[s][0], b), s
        assert np.array_equal(games[s][1], pi), s
        assert np.array_equal(games[s][2], z), s
    assert len(kinds) >= 2


def _games_by_serial(rp):
    """replay dict -> {serial: [(ply, board bytes, counts bytes, player)] sorted by ply}, {serial: z} of finished games"""
    games, z = {}, {}
    for i in np.lexsort((rp["ply"], rp["game_serial"])):
        s = int(rp["game_serial"][i])
        games.setdefault(s, []).append((int(rp["ply"][i]), rp["boards"][i].tobytes(), rp["counts"][i].tobytes(), int(rp["player"][i])))
        if rp["finished"][i]:
            z[s] = float(rp["z"][i])
    return games, z


@pytest.mark.parametrize("evaluator", ["stub", "nn"])
def test_selfplay_rolling_games_do_not_depend_on_the_slot(eng, oracle_mod, evaluator):
    """Rolling self-play (yy_selfplay_advance + yy_selfplay_set_quota): game serial s is the same game -- positions, visit
    counts, Dirichlet noise, sampled actions, result -- whether 40 games are played by 8 slots (5 generations per slot,
    slots restart at different steps) or by 40 slots at once, with a launch boundary in the middle of searches."""
    import torch
    from oracle import port
    n = m = 6
    total, sims = 40, 30
    kw = {}
    if evaluator == "nn":
        torch.manual_seed(11)
        kw["state_dict"] = randomise_bn(port.build_net(n, m, 128, 1)).state_dict()
    runs = []
    for slots, chunk in ((8, 97), (40, 1000)):
        e = eng.Engine(rows=n, cols=m, n_games=slots, n_sims=sims, evaluator=evaluator, seed=77, replay_capacity=total * 400, **kw)
        e.selfplay_set_quota(total)
        for _ in range(4000):
            e.selfplay_advance(chunk)
            st = e.stats()
            if st.games_finished >= total:
                break
        assert st.games_finished == total and st.overflow == 0 and st.examples <= total * 400
        e.selfplay_advance(50)                           # quota used up: every slot idles, nothing more happens
        st2 = e.stats()
        assert (st2.moves, st2.examples, st2.tower_evals) == (st.moves, st.examples, st.tower_evals)
        assert st.tower_evals == st.evals + st.moves     # every evaluated board was a pending leaf (or a root)
        runs.append(_games_by_serial(e.replay()))
        e.close()
    (g8, z8), (g40, z40) = runs
    assert sorted(g8) == list(range(total)) and g8 == g40 and z8 == z40 and len(z8) == total


def test_selfplay_rolling_matches_lockstep_kernels(eng, oracle_mod):
    """The persistent kernel playing the games itself (one launch, slots advance independently) against the lock-step
    driver (prepare / noise / root / per-simulation step / move kernels, YY_MODE_STEP_KERNELS): every (game, ply) that
    both played has the same position, visit counts and mover."""
    n = m = 6
    slots, sims, moves = 24, 40, 45
    runs = []
    for sk in (False, True):
        e = eng.Engine(rows=n, cols=m, n_games=slots, n_sims=sims, evaluator="stub", seed=5, step_kernels=sk)
        e.selfplay_run(moves)
        st = e.stats()
        assert st.moves == slots * moves and st.overflow == 0
        runs.append(_games_by_serial(e.replay()))
        e.close()
    (ga, za), (gb, zb) = runs
    common = 0
    for s in set(ga) & set(gb):
        k = min(len(ga[s]), len(gb[s]))
        assert ga[s][:k] == gb[s][:k], s
        common += k
        if s in za and s in zb:
            assert za[s] == zb[s]
    assert common >= slots * moves // 2


@pytest.mark.parametrize("n,m", [(8, 8), (6, 6), (5, 7), (16, 16), (9, 11)])
def test_device_pack_unpack_matches_host_packing(yy, n, m):
    """yy_pack_boards / yy_unpack_boards (the int8 <-> bitboard conversion of the host-buffer entry points) against the numpy
    packing of bitboard.py, including the last partial word."""
    from yinyang_game_alphazero_b200 import engine, bitboard
    rng = np.random.default_rng(n * 100 + m)
    boards = rng.integers(-1, 2, (700, n, m)).astype(np.int8)
    b, w = engine.pack_boards_dev(boards, n, m)
    hb, hw = bitboard.pack_boards(boards, n, m)
    assert np.array_equal(b.cpu().numpy().view(np.uint64), hb) and np.array_equal(w.cpu().numpy().view(np.uint64), hw)
    back, bits = engine.unpack_boards_dev(n, m, b, w, mask=b)
    assert np.array_equal(back, boards) and np.array_equal(bits, (boards == 1).reshape(700, -1).astype(np.uint8))
    only_mask = engine.unpack_boards_dev(n, m, mask=w)
    assert only_mask[0] is None and np.array_equal(only_mask[1], (boards == -1).reshape(700, -1).astype(np.uint8))
