// yy_dataset.cu -- replay records -> training tensors with the 8-fold symmetry augmentation, on the device.
//
// Restates create_dataset_from_games / DataProcessor.preprocess_sample / augment_sample
// (src/yin_yang/ai/data_utils.py:16-215) over board_to_input (src/yin_yang/ai/neural_network.py:156-196) and
// Node.get_children_distribution at temperature 1 (src/yin_yang/ai/mcts.py:183-215) for a whole replay buffer:
// for every record the input planes [5][n][m] (empty, black, white, row fill, column fill) and the policy [A] are
// written in the 8 forms of augment_sample, in its order (identity, rot90 x1/x2/x3 counter-clockwise, flip left-right,
// flip up-down, transpose, anti-transpose), the value replicated.  All arithmetic is the reference's: fractions are
// float64 quotients rounded to float32 (Python float -> torch.float32), the forms are pure permutations => bit-exact.
//
// Roofline: HBM, write bound.  Algorithmic bytes per record = 16W + 2A + 4 read, 8*(6A + 1)*4 written
// (12,468 B at 8x8).  One warp per record; every store instruction writes 32 consecutive floats.
#include "yy_common.cuh"

namespace yy {

constexpr int kDatasetBlock = 256;   // 8 records per CTA
constexpr int kDatasetWarps = kDatasetBlock / 32;

// One warp per record, two phases.  (1) The six source planes of the record (empty, black, white, row fill, column
// fill, policy) are computed ONCE per cell into the warp's slice of shared memory -- this is where the float64
// quotients are.  (2) The 8 forms are pure permutations of those planes: every output element is one shared-memory
// load and one streaming store (32 consecutive floats per store instruction; the output is written once and far
// exceeds L2).  The first version recomputed the quotients for each of the 8 forms and was bound by FP64 issue, not HBM.
__host__ __device__ inline int dataset_smem_floats(int A) { return 6 * A + 64; }   // per warp: planes + row / column fractions

// M = board side when it is one of the common sizes (all offsets become immediates), 0 = read it from g.
// FORMS = 8: all forms of augment_sample; FORMS = 1: the identity form only (preprocess_sample, any board shape).
template <int NW, int M, int FORMS = 8>
__global__ void __launch_bounds__(kDatasetBlock, 4)
augment_kernel(Geo<NW> g, int W, const uint64_t* __restrict__ black, const uint64_t* __restrict__ white,
               const uint16_t* __restrict__ counts, const float* __restrict__ policy_in, const float* __restrict__ values,
               long long count, float* __restrict__ out_planes, float* __restrict__ out_policy, float* __restrict__ out_values) {
  extern __shared__ float s_dataset[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * kDatasetWarps + warp;
  if (r >= count) return;                       // whole warps leave; only warp-level synchronisation below
  const int n = M ? M : g.rows, m = M ? M : g.cols, A = M ? M * M : g.cells;
  float* src = s_dataset + warp * dataset_smem_floats(A);
  float* rowv = src + 6 * A;                    // [32] fill fraction of row x
  float* colv = rowv + 32;                      // [32] fill fraction of column y
  const BB<NW> b = load_bb<NW>(black, r, W) & g.full, w = load_bb<NW>(white, r, W) & g.full;
  const BB<NW> occ = b | w;
  // row / column fill fractions (neural_network.py:183-194): lane x computes row x's, lane y column y's  (n, m <= 32)
  int rc = 0, cc = 0;
  for (int y = 0; y < m; ++y) rc += (lane < n && test(occ, lane * m + y)) ? 1 : 0;
  for (int x = 0; x < n; ++x) cc += (lane < m && test(occ, x * m + lane)) ? 1 : 0;
  rowv[lane] = (float)((double)rc / (double)m);
  colv[lane] = (float)((double)cc / (double)n);
  // policy = visit counts / their sum in float64 (uniform when there is no visit, mcts.py:209-213), then float32
  unsigned total = 0;
  if (counts) {
    for (int a = lane; a < A; a += 32) total += counts[r * A + a];
    for (int off = 16; off; off >>= 1) total += __shfl_xor_sync(0xffffffffu, total, off);
  }
  const float uniform = (float)(1.0 / (double)A);
  if (lane < FORMS && out_values) out_values[r * FORMS + lane] = values ? values[r] : 0.0f;
  __syncwarp();
  for (int s = lane; s < A; s += 32) {          // phase 1: the identity form, once per cell
    const int sx = s / m, sy = s - sx * m;
    const bool isb = test(b, s), isw = test(w, s);
    src[s] = (isb || isw) ? 0.0f : 1.0f;
    src[A + s] = isb ? 1.0f : 0.0f;
    src[2 * A + s] = isw ? 1.0f : 0.0f;
    src[3 * A + s] = rowv[sx];
    src[4 * A + s] = colv[sy];
    float p;
    if (counts) p = total ? (float)((double)counts[r * A + s] / (double)total) : uniform;
    else p = policy_in[r * A + s];
    src[5 * A + s] = p;
  }
  __syncwarp();
  float* planes0 = out_planes + r * (5ll * FORMS) * A;   // [FORMS][5 planes][A]
  float* pol0 = out_policy + r * (long long)FORMS * A;   // [FORMS][A]
  for (int a = lane; a < A; a += 32) {          // phase 2: output cell a of form f <- source cell form_src(f, a)
#pragma unroll
    for (int f = 0; f < FORMS; ++f) {           // (square boards: n == m)
      const float* sp = src + form_src(f, n, m, a);
      float* planes = planes0 + f * 5 * A + a;
#pragma unroll
      for (int k = 0; k < 5; ++k) __stcs(planes + k * A, sp[k * A]);
      __stcs(pol0 + f * A + a, sp[5 * A]);
    }
  }
}

}  // namespace yy

using namespace yy;

// DataProcessor.preprocess_sample for a whole buffer (data_utils.py:16-37): planes and policy of every record, no
// augmentation -- any board shape (create_dataset_from_games(..., augment=False) on a 5 x 7 board).
extern "C" int yy_dataset_samples(int rows, int cols, const uint64_t* black, const uint64_t* white, const uint16_t* counts,
                                  const float* policy, const float* values, int64_t count, float* out_planes,
                                  float* out_policy, float* out_values, void* stream) {
  if (!board_supported(rows, cols)) return set_error(YY_ERR_INVALID, "unsupported board %dx%d", rows, cols);
  if (count < 0) return set_error(YY_ERR_INVALID, "negative count");
  if (yy_device_count() == 0) return set_error(YY_ERR_NO_DEVICE, "no CUDA device: the engine has no CPU fallback");
  if (count == 0) return YY_OK;
  if (!black || !white || (!counts && !policy) || !out_planes || !out_policy) return set_error(YY_ERR_INVALID, "null argument");
  const int cells = rows * cols, W = words_for_cells(cells);
  const unsigned grid = (unsigned)((count + kDatasetWarps - 1) / kDatasetWarps);
  const size_t smem = (size_t)kDatasetWarps * dataset_smem_floats(cells) * sizeof(float);
#define YY_DATASET_LAUNCH(NWV)                                                                                          \
  do {                                                                                                                  \
    if (smem > 48 * 1024)                                                                                               \
      cudaFuncSetAttribute(augment_kernel<NWV, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
    augment_kernel<NWV, 0, 1><<<grid, kDatasetBlock, smem, (cudaStream_t)stream>>>(                                     \
        make_geo<NWV>(rows, cols, 0), W, black, white, counts, policy, values, count, out_planes, out_policy, out_values); \
  } while (0)
  YY_DISPATCH_NW(cells, YY_DATASET_LAUNCH(NW));
#undef YY_DATASET_LAUNCH
  YY_LAUNCH_CHECK();
  return YY_OK;
}

extern "C" int yy_augment_samples(int rows, int cols, const uint64_t* black, const uint64_t* white, const uint16_t* counts,
                                  const float* policy, const float* values, int64_t count, float* out_planes,
                                  float* out_policy, float* out_values, void* stream) {
  if (!board_supported(rows, cols)) return set_error(YY_ERR_INVALID, "unsupported board %dx%d", rows, cols);
  if (rows != cols) return set_error(YY_ERR_INVALID, "augmentation rotates by 90 degrees: square boards only (data_utils.py:59-76)");
  if (count < 0) return set_error(YY_ERR_INVALID, "negative count");
  if (yy_device_count() == 0) return set_error(YY_ERR_NO_DEVICE, "no CUDA device: the engine has no CPU fallback");
  if (count == 0) return YY_OK;     // empty replay buffer: nothing to write (pointers may be null)
  if (!black || !white || (!counts && !policy) || !out_planes || !out_policy) return set_error(YY_ERR_INVALID, "null argument");
  const int cells = rows * cols, W = words_for_cells(cells);
  const unsigned grid = (unsigned)((count + kDatasetWarps - 1) / kDatasetWarps);
  const size_t smem = (size_t)kDatasetWarps * dataset_smem_floats(cells) * sizeof(float);   // <= 50,176 B at 256 cells
#define YY_AUGMENT_LAUNCH(NWV, MV)                                                                                      \
  do {                                                                                                                  \
    if (smem > 48 * 1024)                                                                                               \
      cudaFuncSetAttribute(augment_kernel<NWV, MV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);            \
    augment_kernel<NWV, MV><<<grid, kDatasetBlock, smem, (cudaStream_t)stream>>>(                                       \
        make_geo<NWV>(rows, cols, 0), W, black, white, counts, policy, values, count, out_planes, out_policy, out_values); \
  } while (0)
  if (rows == 8) YY_AUGMENT_LAUNCH(1, 8);
  else if (rows == 6) YY_AUGMENT_LAUNCH(1, 6);
  else if (rows == 16) YY_AUGMENT_LAUNCH(4, 16);
  else YY_DISPATCH_NW(cells, YY_AUGMENT_LAUNCH(NW, 0));
#undef YY_AUGMENT_LAUNCH
  YY_LAUNCH_CHECK();
  return YY_OK;
}
