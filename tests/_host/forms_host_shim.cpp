// Test-only: compiles the board-form map and the random-form hash of the product's rules header (yy_rules.cuh) for
// the HOST with g++, so that the CPU suite can check them against numpy and the oracle.  Never linked into the product.
#include "../../yinyang-game-alphazero_b200/csrc/yy_rules.cuh"
using namespace yy;

// out[c] = form_src(f, c) for every cell; -1 when f is not a form of a rows x cols board
extern "C" int yyh_form_src(int f, int rows, int cols, int32_t* out) {
  if (!form_valid(f, rows, cols)) return -1;
  for (int c = 0; c < rows * cols; ++c) out[c] = form_src(f, rows, cols, c);
  return 0;
}

template <int NW>
static void hashed(int rows, int cols, const uint64_t* black, const uint64_t* white, long count, uint64_t seed, int32_t* out) {
  Geo<NW> g = make_geo<NW>(rows, cols, 0);
  const int W = (rows * cols + 63) / 64;
  for (long i = 0; i < count; ++i) {
    BB<NW> b = bb_zero<NW>(), w = bb_zero<NW>();
    for (int k = 0; k < W; ++k) { b.w[k] = black[i * W + k]; w.w[k] = white[i * W + k]; }
    out[i] = hashed_form(stub_key(g, b & g.full, w & g.full), seed, rows, cols);
  }
}

// the form random-form evaluation gives each of `count` packed boards under engine seed `seed`
extern "C" int yyh_hashed_form(int rows, int cols, const uint64_t* black, const uint64_t* white, long count, uint64_t seed,
                               int32_t* out) {
  const int cells = rows * cols;
  if (cells <= 64) hashed<1>(rows, cols, black, white, count, seed, out);
  else if (cells <= 128) hashed<2>(rows, cols, black, white, count, seed, out);
  else if (cells <= 256) hashed<4>(rows, cols, black, white, count, seed, out);
  else return -1;
  return 0;
}
