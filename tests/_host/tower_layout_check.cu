// Test-only: the tower's position layouts (yy_tower.cuh) checked on the host.  For a geometry it walks every M row of every
// tile of a full group and verifies the algebra the persistent kernel relies on:
//   1  every (board < Gb, cell) is held by exactly one M row;
//   2  every tap (dy, dx) of a real cell reads the neighbouring cell of the SAME board when that cell is on the board, and a
//      position that never holds a cell (zero padding) when it is not;
//   3  every position touched lies inside the activation region ([-TW_PAD, TW_ROWS - TW_PAD) rows);
//   4  (layouts with tile skew) a tap of a tile never reads a CELL held by another tile (half-board tiles: by another board):
//      tiles / units are independent through the tower, so they may run layers ahead of each other.  (It may read padding
//      rows of a neighbouring tile -- 6x6: the zero column of its last row group -- which every epilogue rewrites as zeros.)
// Returns 0 when everything holds, else a code (1..4) * 1000000 + the offending M row.  Never linked into the product.
#include <vector>
#include <map>
#include "../../yinyang-game-alphazero_b200/csrc/yy_tower.cuh"
using namespace yy;

extern "C" int yyh_tower_layout(int rows, int cols, int* out_layout, int* out_boards_per_group, int* out_tiles, double* out_useful) {
  if (!nn_geometry_ok(rows, cols)) return -1;
  const TowerGeo g = make_tower_geo(rows, cols, 10);
  const int T = tower_tiles_for(g, g.Gb);
  *out_layout = g.row_aligned; *out_boards_per_group = g.Gb; *out_tiles = T;
  *out_useful = (double)g.Gb * g.A / (128.0 * T);
  std::map<int, int> cell_at;            // padded position -> v of the real cell it holds
  std::map<int, int> tile_of;            // padded position -> tile whose M row it is
  std::vector<int> seen((size_t)g.Gb * 256, 0);
  for (int i = 0; i < 128 * T; ++i) {
    int p, v; tower_row(g, i, p, v);
    if (p != tower_tile_start(g, i >> 7) + (g.sbo_bytes == 128 ? (i & 127) : ((i & 127) >> 3) * (g.sbo_bytes / 16) + (i & 7))) return 5000000 + i;   // descriptor walk
    if (TW_PAD + p < 0 || TW_PAD + p >= TW_ROWS) return 3000000 + i;
    tile_of[p] = i >> 7;
    if (v >= 0) { if (seen[v]++) return 1000000 + i; cell_at[p] = v; }
  }
  for (int b = 0; b < g.Gb; ++b) for (int c = 0; c < g.A; ++c) if (seen[b * 256 + c] != 1) return 1000000;
  const bool skew = g.row_aligned == 2 || g.row_aligned == 3 || g.row_aligned == 4;
  for (int i = 0; i < 128 * T; ++i) {
    int p, v; tower_row(g, i, p, v);
    if (v < 0) continue;
    const int b = v >> 8, cell = v & 255, y = cell / g.m, x = cell % g.m, t = i >> 7;
    for (int dy = -1; dy <= 1; ++dy) for (int dx = -1; dx <= 1; ++dx) {
      const int q = p + dy * g.dy_rows + dx;
      if (TW_PAD + q < 0 || TW_PAD + q >= TW_ROWS) return 3000000 + i;
      const bool on = y + dy >= 0 && y + dy < g.n && x + dx >= 0 && x + dx < g.m;
      auto it = cell_at.find(q);
      if (on) { if (it == cell_at.end() || it->second != b * 256 + (y + dy) * g.m + (x + dx)) return 2000000 + i; }
      else if (it != cell_at.end()) return 2000000 + i;
      if (skew) {
        auto tt = tile_of.find(q);
        if (tt != tile_of.end()) {
          const bool same_unit = g.row_aligned == 2 ? (tt->second >> 1) == (t >> 1) : tt->second == t;
          if (!same_unit && cell_at.count(q)) return 4000000 + i;
        }
      }
    }
  }
  return 0;
}

// The choices of the persistent kernel's code paths for a board, as yy_fused.cu makes them: out = layout, group size
// before / after the FC_N clamp, tiles of a full group, policy M tiles, K panels, K stages per head, rows of the last
// policy tile, boards per heads pass.  Returns -1 when the network kernel does not accept the board.
extern "C" int yyh_tower_classes(int rows, int cols, int* out) {
  if (!nn_geometry_ok(rows, cols)) return -1;
  const TowerGeo raw = make_tower_geo(rows, cols, 10);
  const TowerGeo g = make_fused_geo(rows, cols, 10);
  const FcGeo f = make_fc_geo(g.A);
  const int v[9] = {g.row_aligned, raw.Gb, g.Gb, tower_tiles_for(g, g.Gb), f.Tp, f.n_panels, f.KS, f.Rp_last, fused_batch_boards(g)};
  for (int i = 0; i < 9; ++i) out[i] = v[i];
  return 0;
}
