// yy_tower.cuh -- geometry, weight-stream layout and shared-memory map of the tcgen05 residual tower
// (host side: yy_nn.cu; device side: the persistent search kernel in yy_fused.cu).
//
// A CTA walks "groups" of boards.  A group is a flat list of up to 512 padded positions: each board contributes
// (n+1) x (m+1) positions -- its n x m cells plus one zero column on the right and one zero row below -- so that the
// 3x3 tap (dy,dx) of EVERY position is the position dy*(m+1)+dx further along the list and zero padding comes for free.
// The whole residual tower runs with the group's activations resident in shared memory ([C/8 chunks][616 rows][8 ch]
// bf16 = no-swizzle K-major UMMA core matrices, so a tap shift is just a +16 B/row move of the descriptor start
// address); only the weights stream in (K = 64 stages by cp.async.bulk into a 4-deep mbarrier ring, shared by the
// group's 4 M=128 tiles).  For 8-wide boards the MMA's 8-row groups are the board rows themselves (descriptor SBO =
// 9*16 B skips the zero column): 7 boards per group, 87.5 % of the MMA rows are real cells.  Accumulators live in TMEM
// (4 tiles x 128 fp32 columns = all 512 columns).  The skip connection never touches shared memory: conv1's epilogue
// re-loads the block input into the TMEM accumulator (tcgen05.st) before overwriting it in place, and conv2
// accumulates on top of it.  Algorithmic FLOPs per board: 2*A*(9*5*C + blocks*2*9*C*C + C*64) + FC heads.
#pragma once
#include <cuda_bf16.h>

#include "yy_common.cuh"
#include "yy_ptx.cuh"

namespace yy {

constexpr int TW_C = 128;              // tower width the kernel is specialised for (narrower nets are zero-padded)
constexpr int TW_CHUNKS = TW_C / 8;    // 16-byte channel chunks per position
constexpr int TW_HEADC = 64;           // policy 32 + value 32 head-conv channels
constexpr int TW_INC = 16;             // stem input channels after padding (K = 16 per tap)
constexpr int TW_MAXT = 4;             // tiles (of 128 positions) per group
constexpr int TW_PAD = 24;             // zero rows before/after the group's positions (>= m+2)
constexpr int TW_ROWS = 680;            // activation rows: flat 512+2*24, row-aligned 24+64*9+10, half-board 24+2*289+18, interleaved 24+4*162+8
constexpr int TW_STAGES = 3;
constexpr int TW_STAGE_BYTES = 16384;
constexpr int TW_CONV_SLOTS = TW_STAGES;   // the tower's view of the weight ring: whole-tap stages, a CTA's half = 16 KB (measured: 8 KB
constexpr int TW_CONV_SLOT_BYTES = TW_STAGE_BYTES;   // half-tap stages in 6 slots stream SLOWER -- a bulk copy costs ~900 cycles whatever its size)
constexpr int TW_EPI_WARPS = 16;           // one (tile, TMEM-lane-quarter) pair per warp
constexpr int TW_BG_WARPS = 2;             // background selection warps (games whose simulations end without an evaluation)
constexpr int TW_THREADS = 64 + 32 * TW_EPI_WARPS + 32 * TW_BG_WARPS;
constexpr int TW_EPI_THREADS = 32 * TW_EPI_WARPS;

constexpr int SM_ACT = 0;
constexpr int SM_RING = SM_ACT + TW_CHUNKS * TW_ROWS * 16;            // 157696
constexpr int SM_POS = SM_RING + TW_STAGES * TW_STAGE_BYTES;          // position tables: padded position + (board, cell)
constexpr int SM_BAR = SM_POS + 2 * 128 * TW_MAXT * 2;
constexpr int TW_FC_SLOTS = 5;          // weight slots during the FC heads: the ring + 2 in the free tail of the activation region
constexpr int TW_NBAR = 6;              // barrier sets (full, empty, peer-full): max(TW_CONV_SLOTS, TW_FC_SLOTS)
constexpr int TW_FC_EXTRA_OFF = 136 * 1024;   // (the FC feature panel ends at 135,168 B)
constexpr int SM_TMEM = SM_BAR + 8 * (3 * TW_NBAR + 4 + 2 * TW_MAXT);   // full, empty, peer-full per slot + (acc_full, act_ready) per half of a group and per tile
constexpr int SM_BIAS = (SM_TMEM + 16 + 15) & ~15;                                 // current / next layer's 128 fp32 biases (double buffer)
constexpr int SM_CNT = SM_BIAS + 2 * TW_C * 4;            // counts of the CTA (pair): [step parity][cluster rank][pending leaves, selecting]
constexpr int SM_BIAS_T = SM_CNT + 48;                   // 8 counts + the background warps' stop flag; then per-tile bias double buffers (skewed tiles)
constexpr int SM_TOTAL = SM_BIAS_T + TW_MAXT * 2 * TW_C * 4;
constexpr int TW_SKEW = 2;               // stages at the head and at the tail of a layer that the MMA issuer walks tile by tile (<= TW_STAGES)
static_assert(SM_TOTAL <= 232448, "persistent kernel exceeds the 227 KB opt-in shared memory of sm_100");
static_assert(TW_FC_EXTRA_OFF + (TW_FC_SLOTS - TW_STAGES) * TW_STAGE_BYTES <= TW_CHUNKS * TW_ROWS * 16, "FC slots exceed the activation region");

struct TowerGeo {
  int n, m, A, W, pitch, PB;  // PB = padded positions per board
  int T, Gb;                  // tiles per group, boards per group
  int blocks;
  // Two layouts of a group's positions (both keep a zero column right of and a zero row below every board):
  //  flat        : M row r of tile t is padded position t*128 + r            (SBO 128 B, any board width)
  //  row-aligned : (cols == 8) an 8-row MMA group is exactly one board row: M row r of tile t is padded position
  //                (16t + r/8)*pitch + r%8, SBO = pitch*16 B -- the zero column is skipped, 7 boards per 4 tiles
  //  half-board  : (16 x 16, row_aligned == 2) tile t = columns [8(t%2), +8) of board t/2: M row r is padded position
  //                (t/2)*PB + (r/8)*pitch + 8(t%2) + r%8, SBO = pitch*16 B -- neither the zero column nor the zero row
  //                is an MMA row: 2 boards per 4 tiles, 100 % of the MMA rows are real cells
  //  interleaved : (8 x 8, row_aligned == 3) the rows of two boards alternate: row group j of tile t is row j/2 of
  //                board 2t + j%2, at padded position 162t + 9j; two zero row groups separate consecutive pairs and a
  //                vertical tap moves TWO row groups (dy_rows = 18).  No zero row is an MMA row: 8 boards per 4 tiles,
  //                100 % of the MMA rows are real cells (row-aligned: 7 boards, 87.5 %)
  //  interleaved flat : (row_aligned == 4, narrow boards, e.g. 6 x 6) a tile is 128 consecutive padded positions = 128 / pitch
  //                row groups of `pitch` positions (the board row and its zero column); the rows of `ilv` boards alternate
  //                (row group j of tile t is row j / ilv of board ilv * t + j % ilv), a vertical tap moves `ilv` row groups, and
  //                `ilv` zero row groups separate consecutive tiles WITHOUT being MMA rows.  6 x 6: 3 boards per tile, 108 of
  //                128 MMA rows are real cells (84 %; flat: 10 boards per 4 tiles, 70 %)
  int row_aligned, sbo_bytes, tile_adv, rows_per_board, ilv;
  int dy_rows;                // padded positions between vertically adjacent cells (pitch, or 2*pitch when interleaved)
};

// M row i (tile i / 128, row i % 128) of a group -> its padded position p (in 16-byte activation rows after the TW_PAD zero rows)
// and v = board * 256 + cell of the board cell it holds, or -1 when the row is padding (zero column / zero row / slack).
__host__ __device__ inline void tower_row(const TowerGeo& g, int i, int& p, int& v) {
  int b, y, x;
  if (g.row_aligned == 3) {
    const int t = i >> 7, j = (i & 127) >> 3;
    x = i & 7; b = 2 * t + (j & 1); y = j >> 1; p = t * g.tile_adv + j * g.pitch + x;
  } else if (g.row_aligned == 4) {
    const int t = i >> 7, r = i & 127, j = r / g.pitch;
    x = r % g.pitch; y = j / g.ilv; b = g.ilv * t + j % g.ilv; p = t * g.tile_adv + r;
  } else if (g.row_aligned == 2) {
    const int t = i >> 7, r = i & 127;
    b = t >> 1; y = r >> 3; x = 8 * (t & 1) + (r & 7); p = b * g.PB + y * g.pitch + x;
  } else if (g.row_aligned) {
    const int R = (i >> 7) * 16 + ((i & 127) >> 3);
    x = i & 7; p = R * g.pitch + x; b = R / g.rows_per_board; y = R % g.rows_per_board;
  } else {
    p = i; b = p / g.PB; const int rem = p % g.PB; y = rem / g.pitch; x = rem % g.pitch;
  }
  v = (b < g.Gb && y < g.n && x < g.m) ? b * 256 + y * g.m + x : -1;
}
// first padded position of tile t (what the MMA descriptor of the tile starts at)
__host__ __device__ inline int tower_tile_start(const TowerGeo& g, int t) {
  return g.row_aligned == 2 ? (t >> 1) * g.PB + (t & 1) * 8 : t * g.tile_adv;
}
// tiles a group of nb boards needs (flat: + pitch + 1, the taps of the last real position read that far)
__host__ __device__ inline int tower_tiles_for(const TowerGeo& g, int nb) {
  const int t = g.row_aligned == 4 ? ((nb + g.ilv - 1) / g.ilv) : g.row_aligned == 3 ? ((nb + 1) >> 1) : g.row_aligned == 2 ? (2 * nb)
              : g.row_aligned ? ((nb * g.rows_per_board + 15) >> 4) : ((nb * g.PB + g.pitch + 1 + 127) >> 7);
  return t < g.T ? t : g.T;
}

// ---- weight-stream geometry shared by producer and MMA issuer ----
struct LayerInfo { int n_stages, stage_bytes, nk16, N; long long stream_off; };
// `stage_bytes` is what the stream holds per stage; a CTA of a pair (cg = 2) stages half of it (its half of the output
// channels).  Single CTA: a stage is one 64-channel slab of one tap (16 KB).  Pair: a stage is one whole tap (K = 128,
// 2 x 16 KB), so a ring slot still carries 16 KB per CTA and feeds 32 MMAs.
__host__ __device__ inline LayerInfo layer_info(int l, int blocks, int cg = 1) {
  LayerInfo li;
  const long long stem = 9ll * (2 * 128 * 16);
  const long long conv = 18ll * TW_STAGE_BYTES;    // bytes of one 3x3 conv layer, either way
  if (l == 0) { li.n_stages = 9; li.stage_bytes = 2 * 128 * 16; li.nk16 = 1; li.N = 128; li.stream_off = 0; }
  else if (l <= 2 * blocks) {
    li.N = 128; li.stream_off = stem + (long long)(l - 1) * conv;
    if (cg == 2) { li.n_stages = 9; li.stage_bytes = 2 * TW_STAGE_BYTES; li.nk16 = 8; }
    else { li.n_stages = 18; li.stage_bytes = TW_STAGE_BYTES; li.nk16 = 4; }
  } else {
    li.N = TW_HEADC; li.stream_off = stem + (long long)(2 * blocks) * conv;
    if (cg == 2) { li.n_stages = 1; li.stage_bytes = 16 * TW_HEADC * 16; li.nk16 = 8; }
    else { li.n_stages = 2; li.stage_bytes = 8 * TW_HEADC * 16; li.nk16 = 4; }
  }
  return li;
}
__host__ __device__ inline long long conv_stream_bytes(int blocks) {
  LayerInfo li = layer_info(2 * blocks + 1, blocks);
  return li.stream_off + (long long)li.n_stages * li.stage_bytes;
}
// stage j of layer l: which 3x3 tap and which first activation chunk it covers
__device__ __forceinline__ void stage_info(int l, int j, int blocks, int pitch, int dy_rows, int cg, int& tapshift, int& chunk0) {
  int tap, slab;
  if (l == 0) { tap = j; slab = 0; }
  else if (l <= 2 * blocks) { if (cg == 2) { tap = j; slab = 0; } else { tap = j >> 1; slab = j & 1; } }
  else { tap = 4; slab = cg == 2 ? 0 : j; }
  tapshift = (tap / 3 - 1) * dy_rows + (tap % 3 - 1);
  chunk0 = slab * 8;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// ------------------------------------------------------------------------------------------------ host side
struct WeightLayout {
  int64_t conv_stream, conv_bias, fc_policy_w, fc_policy_b, fc_value1_w, fc_value1_b, fc_value2_w, fc_value2_b, total;
  int a_pad;
  int64_t fc_stream, fc_stream_bytes;   // stage-ordered policy FC + value FC1 weights for the persistent kernel
  int64_t conv_stream_pair;             // conv stream with every stage split into two N halves (CTA-pair kernel)
};

// ---- FC heads inside the persistent kernel (yy_fused.cu): out[o][board] = W[o][:] . feat[board][:] as UMMA with the
// weights as the M=128 operand (streamed through the same ring as the conv weights) and up to FC_N boards as N.
constexpr int FC_N = 32;                              // boards per FC batch (UMMA N)
constexpr int FC_LBO = FC_N * 16 + 16;                // K-chunk stride of the feature panel (+16 B: conflict-free scatter)
constexpr int FC_PANEL_STAGES = 32;                   // K = 64 per stage -> K = 2048 per panel (135 KB of the act region)
struct FcGeo {
  int Kh;        // K per head = 32 * A (flatten order c*A + cell, neural_network.py:112,117)
  int KS;        // K = 64 stages per (head, M tile)
  int n_panels;  // feature panels per head
  int Tp;        // policy M tiles (A <= 256 -> 1 or 2); the value head always has 2 (256 hidden units)
  int Rp_last;   // rows of the last policy tile, rounded up to 8
};
__host__ __device__ inline FcGeo make_fc_geo(int A) {
  FcGeo f;
  f.Kh = 32 * A; f.KS = (f.Kh + 63) / 64; f.n_panels = (f.KS + FC_PANEL_STAGES - 1) / FC_PANEL_STAGES;
  f.Tp = (A + 127) / 128; f.Rp_last = ((A - 128 * (f.Tp - 1)) + 7) / 8 * 8;
  return f;
}
// stream order: head (policy, value) > panel > M tile > stage; a stage block is [8 K-chunks][R rows][8] bf16
__host__ __device__ inline long long fc_stream_bytes(int A) {
  const FcGeo f = make_fc_geo(A);
  return (long long)f.KS * 128 * ((f.Tp - 1) * 128 + f.Rp_last + 256);
}
inline int64_t align256(int64_t x) { return (x + 255) & ~(int64_t)255; }
inline WeightLayout weight_layout(int rows, int cols, int blocks) {
  WeightLayout w;
  const int A = rows * cols;
  w.a_pad = (A + 15) / 16 * 16;
  int64_t off = 0;
  w.conv_stream = off; off = align256(off + conv_stream_bytes(blocks));
  w.conv_bias = off; off = align256(off + (int64_t)((2 * blocks + 1) * TW_C + TW_HEADC) * 4);
  w.fc_policy_w = off; off = align256(off + (int64_t)w.a_pad * 32 * A * 2);
  w.fc_policy_b = off; off = align256(off + (int64_t)w.a_pad * 4);
  w.fc_value1_w = off; off = align256(off + (int64_t)256 * 32 * A * 2);
  w.fc_value1_b = off; off = align256(off + 256 * 4);
  w.fc_value2_w = off; off = align256(off + 256 * 4);
  w.fc_value2_b = off; off = align256(off + 4);
  w.fc_stream = off; w.fc_stream_bytes = fc_stream_bytes(A); off = align256(off + w.fc_stream_bytes);
  w.conv_stream_pair = off; off = align256(off + conv_stream_bytes(blocks));
  w.total = off;
  return w;
}

inline bool nn_geometry_ok(int rows, int cols) {
  return rows >= 1 && cols >= 1 && cols + 2 <= TW_PAD && (rows + 1) * (cols + 1) <= 128 * TW_MAXT && rows * cols <= 256;
}

inline TowerGeo make_tower_geo(int rows, int cols, int blocks) {
  TowerGeo g;
  g.n = rows; g.m = cols; g.A = rows * cols; g.W = words_for_cells(g.A); g.pitch = cols + 1; g.PB = (rows + 1) * (cols + 1);
  g.blocks = blocks;
  g.row_aligned = 0; g.sbo_bytes = 128; g.tile_adv = 128; g.rows_per_board = rows + 1; g.dy_rows = g.pitch; g.ilv = 1;
  if (cols == 8 && rows == 8) {                  // interleaved board pairs: one M=128 tile = 2 boards, every MMA row a real cell
    g.row_aligned = 3; g.sbo_bytes = g.pitch * 16; g.tile_adv = 18 * g.pitch; g.dy_rows = 2 * g.pitch;
    g.T = TW_MAXT; g.Gb = 2 * TW_MAXT;
    return g;
  }
  if (cols == 16 && rows == 16) {                // half-board tiles: one M=128 tile = 16 board rows x 8 cells, every MMA row is
    g.row_aligned = 2; g.sbo_bytes = g.pitch * 16; g.tile_adv = 0;   // a real cell; tile t starts at (t/2)*PB + (t%2)*8
    g.T = TW_MAXT; g.Gb = TW_MAXT / 2;
    return g;
  }
  if (cols == 8 && rows + 1 <= 16 * TW_MAXT) {   // one board row == one 8-row MMA group
    g.row_aligned = 1; g.sbo_bytes = g.pitch * 16; g.tile_adv = 16 * g.pitch;
    g.T = TW_MAXT; g.Gb = (16 * TW_MAXT) / (rows + 1);
    if (g.Gb > 127) g.Gb = 127;
    return g;
  }
  double best = -1.0; g.T = TW_MAXT; g.Gb = 1;
  for (int T = 1; T <= TW_MAXT; ++T) {
    int Gb = (128 * T) / g.PB;
    if (Gb < 1) continue;
    if (Gb > 127) Gb = 127;
    double eff = (double)Gb * g.A / (128.0 * T);
    if (eff >= best - 1e-12) { best = eff; g.T = T; g.Gb = Gb; }
  }
  // interleaved flat: the largest number of boards whose rows fit one tile and whose vertical tap stays inside the zero rows
  // in front of the first tile; taken when more of its MMA rows are real cells than in the flat layout
  int ilv = (128 / g.pitch) / rows;
  while (ilv > 0 && ilv * g.pitch + 1 > TW_PAD) --ilv;
  if (ilv > 0 && (double)ilv * g.A / 128.0 > best + 1e-9) {
    const int adv = ilv * rows * g.pitch + ilv * g.pitch;        // the tile's row groups + the zero row groups behind them
    if (TW_PAD + (TW_MAXT - 1) * adv + 128 + ilv * g.pitch + 1 <= TW_ROWS) {
      g.row_aligned = 4; g.ilv = ilv; g.tile_adv = adv; g.dy_rows = ilv * g.pitch; g.T = TW_MAXT; g.Gb = ilv * TW_MAXT;
    }
  }
  return g;
}

// The persistent kernel's geometry: a group holds at most FC_N boards, so that a heads pass takes whole groups.
inline TowerGeo make_fused_geo(int rows, int cols, int blocks) {
  TowerGeo g = make_tower_geo(rows, cols, blocks);
  if (g.Gb > FC_N) g.Gb = FC_N;
  return g;
}
// boards per heads pass of the persistent kernel (whole groups, except possibly the last group of a batch)
inline int fused_batch_boards(const TowerGeo& g) {
  if (g.row_aligned == 4) return FC_N;   // groups of 12 boards: a heads pass takes 12 + 12 + 8 (the last group of a batch may be partial)
  int per = (FC_N / g.Gb) * g.Gb;
  return per > 0 ? per : g.Gb;
}

}  // namespace yy
