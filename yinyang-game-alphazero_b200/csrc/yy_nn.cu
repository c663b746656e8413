// yy_nn.cu -- host side of the policy/value network: packed weight image layout, engine scratch, event profiling.
//
// Network (src/yin_yang/ai/neural_network.py:39-123, eval mode, BatchNorm folded into the convolutions by the host
// packer):  board_to_input (:156-196) -> conv3x3(5->C)+ReLU -> blocks x [conv3x3+ReLU, conv3x3 + skip + ReLU] ->
// {policy: conv1x1(C->32)+ReLU -> FC(32A->A)}, {value: conv1x1(C->32)+ReLU -> FC(32A->256)+ReLU -> FC(256->1) -> tanh};
// predict() applies softmax over all A logits (:152).  The device code is the persistent kernel in yy_fused.cu; the
// shared-memory / weight-stream layout it relies on is described in yy_tower.cuh.
#include <cuda_bf16.h>

#include "yy_nn.cuh"
#include "yy_tower.cuh"

namespace yy {

// ------------------------------------------------------------------------------------------------ host side
int64_t nn_weight_bytes(int rows, int cols, int channels, int blocks) {
  if (!nn_geometry_ok(rows, cols) || channels < 1 || channels > TW_C || blocks < 0)
    return set_error(YY_ERR_INVALID, "network geometry unsupported: %dx%d, %d channels, %d blocks (need cols<=%d, channels<=%d)",
                     rows, cols, channels, blocks, TW_PAD - 2, TW_C);
  return weight_layout(rows, cols, blocks).total;
}

// walk entries per board of the head-feature scratch: one per form when the engine averages over the forms
static int scratch_entries_per_board(const yy_engine_config& cfg) {
  return (cfg.mode_flags & YY_MODE_EVAL_AVERAGE_FORMS) ? form_count(cfg.rows, cfg.cols) : 1;
}

// engine scratch = the head-conv features [max_entries][64*A] bf16 (written and re-read by the same CTA: an L2 round trip)
size_t nn_workspace_bytes(const yy_engine_config& cfg) {
  if (cfg.evaluator != YY_EVAL_NN) return 0;
  const int64_t boards = (int64_t)cfg.n_games * (cfg.leaves_per_step > 0 ? cfg.leaves_per_step : 1);
  return (size_t)align256(boards * scratch_entries_per_board(cfg) * TW_HEADC * cfg.rows * cfg.cols * 2);
}

int nn_init(NNState& nn, const yy_engine_config& cfg, void* scratch) {
  nn = NNState{};
  nn.rows = cfg.rows; nn.cols = cfg.cols; nn.A = cfg.rows * cfg.cols; nn.W = words_for_cells(nn.A);
  nn.channels = cfg.nn_channels; nn.blocks = cfg.nn_blocks;
  nn.max_boards = cfg.n_games * (cfg.leaves_per_step > 0 ? cfg.leaves_per_step : 1); nn.device = cfg.device;
  nn.max_entries = nn.max_boards * scratch_entries_per_board(cfg);
  if (cfg.evaluator != YY_EVAL_NN) return YY_OK;
  if (!nn_geometry_ok(cfg.rows, cfg.cols) || cfg.nn_channels > TW_C)
    return set_error(YY_ERR_INVALID, "network geometry unsupported: %dx%d, %d channels", cfg.rows, cfg.cols, cfg.nn_channels);
  nn.scratch = scratch; nn.scratch_bytes = (int64_t)nn_workspace_bytes(cfg);
  YY_CUDA_OK(cudaDeviceGetAttribute(&nn.num_sms, cudaDevAttrMultiProcessorCount, cfg.device));
  int major = 0;
  YY_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, cfg.device));
  if (major != 10) return set_error(YY_ERR_NO_DEVICE, "the inference kernels are sm_100a-only (device reports sm_%d*)", major);
  nn.attrs_set = true;
  return YY_OK;
}
static int nn_drain_events(NNState& nn) {
  for (int i = 0; i < nn.ev_used; ++i) {
    YY_CUDA_OK(cudaEventSynchronize(nn.ev[2 * i + 1]));
    float ms = 0.0f;
    YY_CUDA_OK(cudaEventElapsedTime(&ms, nn.ev[2 * i], nn.ev[2 * i + 1]));
    nn.tower_ms += ms;
  }
  nn.ev_used = 0;
  return YY_OK;
}
void nn_destroy(NNState& nn) {
  if (nn.ev) { for (int i = 0; i < 2 * nn.ev_cap; ++i) cudaEventDestroy(nn.ev[i]); delete[] nn.ev; nn.ev = nullptr; }
}
int nn_set_profiling(NNState& nn, int enable) {
  if (enable && !nn.ev) {
    nn.ev_cap = 1024;
    nn.ev = new cudaEvent_t[2 * nn.ev_cap];
    for (int i = 0; i < 2 * nn.ev_cap; ++i) YY_CUDA_OK(cudaEventCreate(&nn.ev[i]));
  }
  nn.profiling = enable != 0; nn.ev_used = 0; nn.tower_launches = 0; nn.tower_ms = 0.0; nn.tower_boards = 0;
  return YY_OK;
}
int nn_get_profile(NNState& nn, long long* launches, double* total_ms, long long* boards) {
  int rc = nn_drain_events(nn); if (rc) return rc;
  if (launches) *launches = nn.tower_launches;
  if (total_ms) *total_ms = nn.tower_ms;
  if (boards) *boards = nn.tower_boards;
  return YY_OK;
}

int nn_load_weights(NNState& nn, const void* weights, int64_t bytes) {
  int64_t need = nn_weight_bytes(nn.rows, nn.cols, nn.channels, nn.blocks);
  if (need < 0) return (int)need;
  if (!weights || bytes < need) return set_error(YY_ERR_INVALID, "weight image too small: %lld < %lld", (long long)bytes, (long long)need);
  if (((uintptr_t)weights & 255) != 0) return set_error(YY_ERR_INVALID, "weight image must be 256-byte aligned");
  nn.weights = weights; nn.weight_bytes = bytes;
  return YY_OK;
}

}  // namespace yy

// Section offsets of the packed weight image, for the host-side packer:
// out[0..8] = conv_stream, conv_bias, fc_policy_w, fc_policy_b, fc_value1_w, fc_value1_b, fc_value2_w, fc_value2_b, total;
// out[9] = padded policy rows (A rounded up to 16); out[10], out[11] = offset / bytes of the stage-ordered FC stream;
// out[12] = conv stream with N-halved stages (CTA-pair kernel).
extern "C" int yy_nn_weight_layout(int rows, int cols, int channels, int blocks, int64_t* out) {
  using namespace yy;
  int64_t t = nn_weight_bytes(rows, cols, channels, blocks);
  if (t < 0) return (int)t;
  WeightLayout w = weight_layout(rows, cols, blocks);
  out[0] = w.conv_stream; out[1] = w.conv_bias; out[2] = w.fc_policy_w; out[3] = w.fc_policy_b; out[4] = w.fc_value1_w;
  out[5] = w.fc_value1_b; out[6] = w.fc_value2_w; out[7] = w.fc_value2_b; out[8] = w.total; out[9] = w.a_pad;
  out[10] = w.fc_stream; out[11] = w.fc_stream_bytes; out[12] = w.conv_stream_pair;
  return YY_OK;
}
