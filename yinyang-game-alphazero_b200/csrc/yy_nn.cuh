// yy_nn.cuh -- policy/value network inference on the leaf batch (interface used by yy_tree.cu).
// Implementation and memory layouts: yy_nn.cu.
#pragma once
#include "yy_common.cuh"

namespace yy {

struct NNState {
  int rows, cols, A, W, channels, blocks;
  int max_boards;            // boards per launch (>= n_games)
  int max_entries;           // capacity of the head-feature scratch in walk entries (max_boards x forms when averaging)
  const void* weights;       // packed image (device), owned by the caller
  int64_t weight_bytes;
  void* scratch;             // head features etc. (inside the engine workspace)
  int64_t scratch_bytes;
  int device, num_sms;
  bool attrs_set;
  // optional CUDA-event timing of the persistent kernel launches (bench.py's live roofline figure)
  bool profiling;
  cudaEvent_t* ev;           // 2 * ev_cap events
  int ev_cap, ev_used;
  long long tower_launches; double tower_ms; long long tower_boards;
  long long* dbg;            // device buffer for per-layer clock stamps (developer tool), usually nullptr
  int dbg_flags;             // developer A/B switches (yy_engine_set_debug_stamps): bit 0 = ping-pong of group halves
};

int64_t nn_weight_bytes(int rows, int cols, int channels, int blocks);
size_t nn_workspace_bytes(const yy_engine_config& cfg);
int nn_init(NNState& nn, const yy_engine_config& cfg, void* scratch);
void nn_destroy(NNState& nn);
int nn_load_weights(NNState& nn, const void* weights_dev, int64_t bytes);
int nn_set_profiling(NNState& nn, int enable);
// drains recorded event pairs (synchronises) and returns totals since profiling was enabled
int nn_get_profile(NNState& nn, long long* launches, double* total_ms, long long* boards);
struct EngineDev;
// Persistent kernel (yy_fused.cu): up to `iterations` x (network forward on the pending leaves -> heads -> tree step) in
// ONE launch.
//   YY_FUSED_FORWARD  (dev == nullptr): one plain forward of boards [0, count) into policy/value/logits.
//   YY_FUSED_SEARCH   whole search over the engine's leaf batch (slot = game); ends when no game has a pending leaf.
//   YY_FUSED_SELFPLAY rolling self-play: a game whose search is complete makes its move and roots its next search in
//                     the same step (sp_advance_game), within its move budget and the game quota.
// use_nn = false runs the deterministic-prior evaluator (tree steps only).
enum { YY_FUSED_FORWARD = 0, YY_FUSED_SEARCH = 1, YY_FUSED_SELFPLAY = 2 };
// Symmetric evaluation: the dihedral form (form_src, yy_rules.cuh) the network sees a board in.
//   IDENTITY  the board as it is;  FIXED  form `form` for every board;  HASHED  form hashed_form(stub_key(board), seed);
//   AVERAGE   every valid form, policy and value averaged over them (fp32, ascending form order; no logits).
enum { YY_FORM_IDENTITY = 0, YY_FORM_FIXED = 1, YY_FORM_HASHED = 2, YY_FORM_AVERAGE = 3 };
struct FormSpec {
  int mode = YY_FORM_IDENTITY;
  int form = 0;
  uint64_t seed = 0;
};
// walk entries (head-feature rows) per board under a form mode
inline int form_entries(int mode, int rows, int cols) { return mode == YY_FORM_AVERAGE ? form_count(rows, cols) : 1; }
int nn_fused_run(NNState& nn, const EngineDev* dev, uint32_t rule_flags, const uint64_t* black, const uint64_t* white,
                 int64_t count, float* policy, float* value, float* logits, int iterations, bool use_nn, int mode,
                 const FormSpec& forms, cudaStream_t stream);

}  // namespace yy
