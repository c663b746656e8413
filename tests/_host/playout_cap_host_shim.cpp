// Test-only: compiles the playout-cap decision of the product's rules header (yy_rules.cuh: playout_full) for the HOST
// with g++, so that the CPU suite can check it against the Python restatement.  Never linked into the product.
#include "../../yinyang-game-alphazero_b200/csrc/yy_rules.cuh"
using namespace yy;

// out[i] = playout_full(seed, serial[i], ply[i], threshold)
extern "C" void yyh_playout_full(uint64_t seed, const int32_t* serial, const int32_t* ply, long count, uint64_t threshold,
                                 uint8_t* out) {
  for (long i = 0; i < count; ++i) out[i] = playout_full(seed, serial[i], ply[i], threshold) ? 1 : 0;
}
