// yy_rules.cuh -- Yin-Yang rules on bitboards (one thread per board).
//
// Restates, on packed bitboards, the legality predicate of the reference
//   YinYangLogic.is_valid_move      src/yin_yang/yin_yang_logic.py:31-56
//   _check_connectivity             :58-94     (same-colour 4-connectivity)
//   _check_2x2_constraint           :96-109    (no mono-colour 2x2 anywhere)
//   checkRowColumnConstraint        src/gui/static/js/yin_yang_game.js:338-384 (optional flag)
// in closed form (no trial placement):
//   legal(c) = empty(c) AND no existing 2x2 in either colour
//              AND c touches every 4-connected component of the mover's stones (vacuous if none)
//              AND no 2x2 window through c already has its other three cells in the mover's colour.
// Cell (x,y) = bit a = x*cols + y of an NW-word little-endian bit vector.
//
// The functions are __host__ __device__ so that tests/ can compile this header with g++ and
// check the algorithm on the CPU box; the product only ever runs them inside CUDA kernels.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define YY_HD __host__ __device__ __forceinline__
#else
#define YY_HD inline
#endif

#define YY_RULE_ROWCOL_BIT 1u

namespace yy {

YY_HD int popc64(uint64_t x) {
#if defined(__CUDA_ARCH__)
  return __popcll(x);
#else
  return __builtin_popcountll(x);
#endif
}
YY_HD int ctz64(uint64_t x) {
#if defined(__CUDA_ARCH__)
  return __ffsll((long long)x) - 1;
#else
  return __builtin_ctzll(x);
#endif
}

template <int NW>
struct BB {
  uint64_t w[NW];
};

template <int NW> YY_HD BB<NW> bb_zero() { BB<NW> r; for (int i = 0; i < NW; ++i) r.w[i] = 0; return r; }
template <int NW> YY_HD BB<NW> operator&(BB<NW> a, BB<NW> b) { for (int i = 0; i < NW; ++i) a.w[i] &= b.w[i]; return a; }
template <int NW> YY_HD BB<NW> operator|(BB<NW> a, BB<NW> b) { for (int i = 0; i < NW; ++i) a.w[i] |= b.w[i]; return a; }
template <int NW> YY_HD BB<NW> andnot(BB<NW> a, BB<NW> b) { for (int i = 0; i < NW; ++i) a.w[i] &= ~b.w[i]; return a; }
template <int NW> YY_HD bool any(BB<NW> a) { uint64_t o = 0; for (int i = 0; i < NW; ++i) o |= a.w[i]; return o != 0; }
template <int NW> YY_HD bool same(BB<NW> a, BB<NW> b) { uint64_t o = 0; for (int i = 0; i < NW; ++i) o |= a.w[i] ^ b.w[i]; return o == 0; }
template <int NW> YY_HD int popcount(BB<NW> a) { int c = 0; for (int i = 0; i < NW; ++i) c += popc64(a.w[i]); return c; }
// The word is picked by a chain of selects, not by indexing: a run-time index would put the board in local memory.
template <int NW> YY_HD bool test(const BB<NW>& a, int bit) {
  uint64_t word = a.w[0];
  for (int i = 1; i < NW; ++i) word = (bit >> 6) == i ? a.w[i] : word;
  return (word >> (bit & 63)) & 1ull;
}
template <int NW> YY_HD void setbit(BB<NW>& a, int bit) {
  const uint64_t one = 1ull << (bit & 63);
  for (int i = 0; i < NW; ++i) a.w[i] |= (bit >> 6) == i ? one : 0ull;
}
// lowest set bit as a one-bit board (a must be non-zero)
template <int NW> YY_HD BB<NW> lowest(BB<NW> a) {
  BB<NW> r = bb_zero<NW>();
  for (int i = 0; i < NW; ++i)
    if (a.w[i]) { r.w[i] = a.w[i] & (0 - a.w[i]); break; }
  return r;
}
// index of the k-th (0-based) set bit; -1 if fewer
template <int NW> YY_HD int kth_bit(BB<NW> a, int k) {
  for (int i = 0; i < NW; ++i) {
    int c = popc64(a.w[i]);
    if (k < c) {
      uint64_t x = a.w[i];
      for (int j = 0; j < k; ++j) x &= x - 1;
      return i * 64 + ctz64(x);
    }
    k -= c;
  }
  return -1;
}
// shifts by 1 <= k <= 63 across words
template <int NW> YY_HD BB<NW> shl(BB<NW> a, int k) {
  BB<NW> r;
  for (int i = NW - 1; i >= 0; --i) r.w[i] = (a.w[i] << k) | (i > 0 ? (a.w[i - 1] >> (64 - k)) : 0ull);
  return r;
}
template <int NW> YY_HD BB<NW> shr(BB<NW> a, int k) {
  BB<NW> r;
  for (int i = 0; i < NW; ++i) r.w[i] = (a.w[i] >> k) | (i + 1 < NW ? (a.w[i + 1] << (64 - k)) : 0ull);
  return r;
}

// Board geometry: precomputed on the host, passed to kernels by value.
template <int NW>
struct Geo {
  int rows, cols, cells;
  uint32_t rule_flags;
  BB<NW> full;      // all cells
  BB<NW> not_col0;  // cells with y > 0
  BB<NW> not_colL;  // cells with y < cols-1
  BB<NW> row0;      // cells of row 0
  BB<NW> col0;      // cells of column 0
};

template <int NW>
inline Geo<NW> make_geo(int rows, int cols, uint32_t rule_flags) {
  Geo<NW> g;
  g.rows = rows; g.cols = cols; g.cells = rows * cols; g.rule_flags = rule_flags;
  g.full = g.not_col0 = g.not_colL = g.row0 = g.col0 = bb_zero<NW>();
  for (int x = 0; x < rows; ++x)
    for (int y = 0; y < cols; ++y) {
      int a = x * cols + y;
      setbit(g.full, a);
      if (y > 0) setbit(g.not_col0, a);
      if (y < cols - 1) setbit(g.not_colL, a);
      if (x == 0) setbit(g.row0, a);
      if (y == 0) setbit(g.col0, a);
    }
  return g;
}

// neighbour maps: bit c of east(X) is set iff the cell to the WEST of c... no: named by data motion.
//   toE(X): X moved one column to the east  (bit c set iff c's west neighbour is in X)
template <int NW> YY_HD BB<NW> toE(const Geo<NW>& g, BB<NW> x) { return shl(x, 1) & g.not_col0; }
template <int NW> YY_HD BB<NW> toW(const Geo<NW>& g, BB<NW> x) { return shr(x, 1) & g.not_colL; }
template <int NW> YY_HD BB<NW> toS(const Geo<NW>& g, BB<NW> x) { return shl(x, g.cols) & g.full; }
template <int NW> YY_HD BB<NW> toN(const Geo<NW>& g, BB<NW> x) { return shr(x, g.cols); }
template <int NW> YY_HD BB<NW> dilate4(const Geo<NW>& g, BB<NW> x) { return toE(g, x) | toW(g, x) | toS(g, x) | toN(g, x); }

// _check_2x2_constraint (yin_yang_logic.py:96-109) for one colour: some window fully inside X?
template <int NW> YY_HD bool has_2x2(const Geo<NW>& g, BB<NW> x) {
  BB<NW> h = x & toW(g, x);      // c and its east neighbour
  return any(h & toN(g, h));     // ... and the row below
}

// cells c (not in X) such that placing at c completes a 2x2 of X
template <int NW> YY_HD BB<NW> completes_2x2(const Geo<NW>& g, BB<NW> x) {
  BB<NW> e = toW(g, x);  // c's east neighbour in X
  BB<NW> w = toE(g, x);  // c's west neighbour in X
  BB<NW> s = toN(g, x);  // c's south neighbour in X
  BB<NW> n = toS(g, x);  // c's north neighbour in X
  BB<NW> se = toN(g, e), sw = toN(g, w), ne = toS(g, e), nw = toS(g, w);
  return (e & s & se) | (w & s & sw) | (e & n & ne) | (w & n & nw);
}

// 4-connected component of `seed` inside `x` (_check_connectivity BFS, yin_yang_logic.py:58-94).
// Two dilation steps per convergence test (the fixed point is unchanged; at most one step is wasted).
template <int NW> YY_HD BB<NW> flood(const Geo<NW>& g, BB<NW> seed, BB<NW> x) {
  BB<NW> f = seed;
  for (;;) {
    BB<NW> n1 = f | (dilate4(g, f) & x);
    BB<NW> n2 = n1 | (dilate4(g, n1) & x);
    if (same(n2, f)) return f;
    f = n2;
  }
}

// cells adjacent to EVERY component of x (all cells if x is empty)
template <int NW> YY_HD BB<NW> touches_all_components(const Geo<NW>& g, BB<NW> x) {
  BB<NW> acc = g.full, rem = x;
  while (any(rem) && any(acc)) {
    BB<NW> comp = flood(g, lowest(rem), x);
    acc = acc & dilate4(g, comp);
    rem = andnot(rem, comp);
  }
  return acc;
}

// Row/column rule (JS): does board (p,o) already hold a full single-colour row or column?
template <int NW> YY_HD bool rowcol_violated(const Geo<NW>& g, BB<NW> p, BB<NW> o) {
  BB<NW> occ = p | o;
  BB<NW> rm = g.row0;
  for (int x = 0; x < g.rows; ++x) {
    if (same(occ & rm, rm) && (!any(p & rm) || !any(o & rm))) return true;
    rm = shl(rm, g.cols);
  }
  BB<NW> cm = g.col0;
  for (int y = 0; y < g.cols; ++y) {
    if (same(occ & cm, cm) && (!any(p & cm) || !any(o & cm))) return true;
    cm = shl(cm, 1);
  }
  return false;
}
// cells c such that placing the mover's stone (colour p) at c completes a single-colour row/column
template <int NW> YY_HD BB<NW> completes_rowcol(const Geo<NW>& g, BB<NW> p, BB<NW> o) {
  BB<NW> empty = andnot(g.full, p | o), bad = bb_zero<NW>();
  BB<NW> rm = g.row0;
  for (int x = 0; x < g.rows; ++x) {
    BB<NW> e = empty & rm;
    if (popcount(e) == 1 && !any(o & rm)) bad = bad | e;
    rm = shl(rm, g.cols);
  }
  BB<NW> cm = g.col0;
  for (int y = 0; y < g.cols; ++y) {
    BB<NW> e = empty & cm;
    if (popcount(e) == 1 && !any(o & cm)) bad = bad | e;
    cm = shl(cm, 1);
  }
  return bad;
}

// get_valid_moves (yin_yang_logic.py:111-120) without the connectivity test: empty cells that pass the 2x2 rule
// (and the optional row/column rule) for the colour whose stones are `p` (opponent stones `o`).
template <int NW> YY_HD BB<NW> legal_candidates(const Geo<NW>& g, BB<NW> p, BB<NW> o) {
  if (has_2x2(g, p) || has_2x2(g, o)) return bb_zero<NW>();
  BB<NW> cand = andnot(andnot(g.full, p | o), completes_2x2(g, p));
  if (g.rule_flags & YY_RULE_ROWCOL_BIT) {
    if (rowcol_violated(g, p, o)) return bb_zero<NW>();
    cand = andnot(cand, completes_rowcol(g, p, o));
  }
  return cand;
}

// get_valid_moves: legal placements for the colour whose stones are `p` (opponent stones `o`).
template <int NW> YY_HD BB<NW> legal_moves(const Geo<NW>& g, BB<NW> p, BB<NW> o) {
  BB<NW> cand = legal_candidates(g, p, o);
  if (!any(cand)) return cand;
  return cand & touches_all_components(g, p);
}

template <int NW> YY_HD BB<NW> legal_for(const Geo<NW>& g, BB<NW> black, BB<NW> white, int player) {
  return player == 1 ? legal_moves(g, black, white) : legal_moves(g, white, black);
}

// getNextState (yin_yang_game.py:39-58): place if legal, else silent no-op.  Returns true if placed.
template <int NW> YY_HD bool apply_action(const Geo<NW>& g, BB<NW>& black, BB<NW>& white, int player, int action) {
  if (action < 0 || action >= g.cells) return false;
  BB<NW> lm = legal_for(g, black, white, player);
  if (!test(lm, action)) return false;
  if (player == 1) setbit(black, action); else setbit(white, action);
  return true;
}

// getGameEnded (yin_yang_game.py:80-110) given the mover's mask when already known.
// codes: 0 ongoing, 1 win, -1 loss, 2 draw (host maps 2 -> +0.0001).
template <int NW> YY_HD int ended_code_with_mask(const Geo<NW>& g, BB<NW> black, BB<NW> white, int player,
                                                 BB<NW> mover_mask) {
  if (any(mover_mask)) return 0;
  if (any(legal_for(g, black, white, -player))) return 0;
  int bc = popcount(black), wc = popcount(white);
  if (bc > wc) return player == 1 ? 1 : -1;
  if (wc > bc) return player == -1 ? 1 : -1;
  return 2;
}
template <int NW> YY_HD int ended_code(const Geo<NW>& g, BB<NW> black, BB<NW> white, int player) {
  return ended_code_with_mask(g, black, white, player, legal_for(g, black, white, player));
}

// ---- deterministic hash-stub evaluator (specification shared with oracle/yy_oracle.c) ----
YY_HD uint64_t mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
template <int NW> YY_HD uint64_t stub_key(const Geo<NW>& g, BB<NW> black, BB<NW> white) {
  int words = (g.cells + 63) >> 6;
  uint64_t key = 0x243F6A8885A308D3ull;
  for (int i = 0; i < words; ++i) key = mix64(key ^ black.w[i]);
  for (int i = 0; i < words; ++i) key = mix64(key ^ white.w[i]);
  return key;
}
YY_HD float stub_prior(uint64_t key, int a) {
  return (float)(1u + (uint32_t)(mix64(key + 0xD1B54A32D192ED03ull * (uint64_t)(a + 1)) >> 52)) * (1.0f / 65536.0f);
}
YY_HD float stub_value(uint64_t key) {
  return (float)((int32_t)(mix64(key ^ 0xA0761D6478BD642Full) >> 47) - 65536) * (1.0f / 65536.0f);
}

// ---- the dihedral forms of a board, in augment_sample's order (data_utils.py:59-76): 0 identity, 1-3 rot90 x1/x2/x3
// counter-clockwise, 4 flip left-right, 5 flip up-down, 6 transpose, 7 anti-transpose.  Form f of a board S shows at
// cell c the cell form_src(f, c) of S.  The training data (yy_dataset.cu) and the network's symmetric evaluation
// (yy_fused.cu: the stem reads S[form_src(f, c)], output c is the prior of action form_src(f, c)) share this map.
// A rectangular board keeps its shape only under forms 0, 2, 4, 5.
YY_HD int form_count(int rows, int cols) { return rows == cols ? 8 : 4; }
YY_HD int form_at(int k, int rows, int cols) { return rows == cols ? k : (k < 2 ? 2 * k : k + 2); }   // k-th valid form
YY_HD bool form_valid(int f, int rows, int cols) {
  return f >= 0 && f < 8 && (rows == cols || f == 0 || f == 2 || f == 4 || f == 5);
}
YY_HD int form_src(int f, int n, int m, int c) {
  const int i = c / m, j = c - i * m;
  int sx, sy;
  switch (f) {
    case 0: sx = i; sy = j; break;
    case 1: sx = j; sy = m - 1 - i; break;             // np.rot90(S, 1)[i][j] = S[j][m-1-i]
    case 2: sx = n - 1 - i; sy = m - 1 - j; break;     // rot90 x2
    case 3: sx = n - 1 - j; sy = i; break;             // rot90 x3
    case 4: sx = i; sy = m - 1 - j; break;             // flip left-right
    case 5: sx = n - 1 - i; sy = j; break;             // flip up-down
    case 6: sx = j; sy = i; break;                     // transpose
    default: sx = n - 1 - j; sy = m - 1 - i; break;    // flip(transpose, both axes)
  }
  return sx * m + sy;
}
// form of a position under random-form evaluation: a pure function of (engine seed, position)
YY_HD int hashed_form(uint64_t key, uint64_t seed, int rows, int cols) {
  return form_at((int)(mix64(key ^ seed) % (uint64_t)form_count(rows, cols)), rows, cols);
}

// ---- playout cap randomisation of self-play: the search of game `serial` at ply `ply` is a full one iff this holds
// (threshold = llround(p_full * 2^32); 2^32 = always, 0 = never).  A pure function of (engine seed, serial, ply).
YY_HD bool playout_full(uint64_t seed, int serial, int ply, uint64_t threshold) {
  const uint64_t key = mix64(mix64(seed ^ 0x706c61796f757463ull) ^ (((uint64_t)(uint32_t)serial << 20) | (uint64_t)(uint32_t)ply));
  return (key >> 32) < threshold;
}

}  // namespace yy
