// yy_tree.cu -- HBM-resident batched MCTS (one warp per game) + self-play episode driver.
//
// Restates src/yin_yang/ai/mcts.py (Node.expand :50-91, select_child :97-145, update :147-156,
// MCTS.search :275-343, _simulate :345-414) for n_games independent trees at once, and
// SelfPlayWorker.play_game (src/yin_yang/ai/self_play.py:72-192) as device kernels.
//
// Exactness contract (deterministic mode): simulations of one game are strictly sequential (one leaf
// per game per step, no virtual loss), PUCT is evaluated in the reference's numpy>=2 float32 operation
// order with explicit round-to-nearest intrinsics (no FMA contraction), ties resolve to the lowest
// action index (strict '>' scan in ascending action order) => root visit counts are bit-identical to
// the unmodified reference driven through a value-semantics Game adapter (tests/golden/mcts_*.npz).
//
// Roofline: HBM (latency-bound pointer chasing in practice).  Algorithmic bytes per simulation:
// sum over levels of 12*A_l (N,W,P per child read) + 17*A_leaf (edge slots written) + 8 per path edge
// (N,W read-modify-write) + 2*16*W node state -- ~1.5-4 KB at 8x8 (SURVEY 8d).
#include "yy_selfplay_dev.cuh"
#include "yy_nn.cuh"

#include <new>

namespace yy {

constexpr int kTreeBlock = 128;  // 4 games per CTA

// MCTS.search prologue (mcts.py:288-292): fresh tree per game, root = node 0, pending leaf = root (slot g*K).
// A plain search runs n_sims simulations; the lock-step self-play driver (`prepared`) keeps the budget sp_prepare_kernel
// chose (playout cap).
template <int NW>
__global__ void __launch_bounds__(kTreeBlock) tree_root_kernel(EngineDev e, Geo<NW> g, int prepared) {
  int gi = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (gi >= e.n_games) return;
  tree_root_game<NW>(e, g, gi, lane, prepared ? e.g_sim_budget[gi] : e.n_sims);
  if (lane == 0) e.sp_phase[gi] = 0;      // the tree no longer belongs to a rolling self-play search (sp_advance_game)
  if (gi == 0 && lane == 0) { e.active_count[0] = e.n_games; e.active_count[1] = 0; }
}

// One lock-step of every tree (see tree_step_game, yy_tree_dev.cuh); one warp per game.
template <int NW>
__global__ void __launch_bounds__(kTreeBlock) tree_step_kernel(EngineDev e, Geo<NW> g, int parity) {
  int gi = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (gi >= e.n_games) return;
  // pending-leaf counter is double buffered: this step counts into [parity] and clears the other one for the next step
  if (gi == 0 && lane == 0) e.active_count[parity ^ 1] = 0;
  tree_step_game<NW>(e, g, gi, lane, e.active_count + parity);
}

// root.get_children_visit_counts (mcts.py:168-181) + child value sums
__global__ void tree_counts_kernel(EngineDev e, int32_t* counts, float* child_w) {
  int gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= e.n_games) return;
  for (int a = 0; a < e.A; ++a) { counts[(long long)gi * e.A + a] = 0; if (child_w) child_w[(long long)gi * e.A + a] = 0.0f; }
  const long long nb = (long long)gi * e.max_nodes, eb = (long long)gi * e.edges_cap;
  if (!(e.node_flags[nb] & NODE_EXPANDED)) return;
  int base = e.node_edge_base[nb], cnt = e.node_n_edges[nb];
  for (int k = 0; k < cnt; ++k) {
    int a = e.edge_action[eb + base + k];
    counts[(long long)gi * e.A + a] = e.edge_N[eb + base + k];
    if (child_w) child_w[(long long)gi * e.A + a] = e.edge_W[eb + base + k];
  }
}


// stub evaluator on an arbitrary batch (yy_evaluate in YY_EVAL_STUB mode)
template <int NW>
__global__ void stub_eval_kernel(Geo<NW> g, int W, const uint64_t* black, const uint64_t* white, long long count,
                                 float* policy, float* value) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  BB<NW> b = load_bb<NW>(black, i, W) & g.full, w = load_bb<NW>(white, i, W) & g.full;
  uint64_t key = stub_key(g, b, w);
  for (int a = 0; a < g.cells; ++a) policy[i * g.cells + a] = stub_prior(key, a);
  value[i] = stub_value(key);
}

// ------------------------------------------------------------------------------------------------ self-play
// Lock-step episode driver (one thread per game; the device functions live in yy_selfplay_dev.cuh).  Used when the
// search runs as per-step kernels (YY_MODE_STEP_KERNELS, leaves_per_step > 1); otherwise the persistent kernel plays
// the games itself (yy_fused.cu, sp_advance_game).
template <int NW>
__global__ void __launch_bounds__(128) sp_prepare_kernel(EngineDev e, Geo<NW> g) {
  int gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= e.n_games) return;
  const int budget = sp_prepare_one<NW>(e, g, gi);
  e.g_sim_budget[gi] = budget >= 0 ? budget : e.n_sims;     // read by the root kernel of this move's search
}
template <int NW>
__global__ void __launch_bounds__(128) sp_noise_kernel(EngineDev e, Geo<NW> g) {
  int gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= e.n_games) return;
  sp_noise_one<NW>(e, g, gi);
}
template <int NW>
__global__ void __launch_bounds__(128) sp_move_kernel(EngineDev e, Geo<NW> g) {
  int gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= e.n_games) return;
  sp_move_one<NW>(e, g, gi);
}
__global__ void sp_budget_kernel(EngineDev e, int moves) {
  int gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi < e.n_games) e.sp_moves_left[gi] = moves;
}

__global__ void sp_reset_kernel(EngineDev e) {
  int gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi == 0) { *e.sp_next_serial = 0; Stats z = {}; *e.stats = z; }
  if (gi >= e.n_games) return;
  e.sp_new_game[gi] = 1; e.sp_serial[gi] = -1; e.sp_step[gi] = 0; e.sp_passes[gi] = 0; e.sp_player[gi] = 1;
  e.sp_phase[gi] = 0; e.sp_moves_left[gi] = 0; e.g_npending[gi] = 0;
  for (int k = 0; k < e.W; ++k) { e.sp_black[(long long)gi * e.W + k] = 0; e.sp_white[(long long)gi * e.W + k] = 0; }
}

// ------------------------------------------------------------------------------------------------ host side
struct Carver {
  char* base; size_t off;
  template <typename T> T* take(size_t n) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

static int normalise_cfg(yy_engine_config& c) {
  if (!board_supported(c.rows, c.cols)) return set_error(YY_ERR_INVALID, "unsupported board %dx%d", c.rows, c.cols);
  if (c.n_games < 1 || c.n_sims < 0) return set_error(YY_ERR_INVALID, "n_games >= 1 and n_sims >= 0 required");
  if (c.n_sims > 65000) return set_error(YY_ERR_INVALID, "n_sims must be <= 65000 (16-bit node ids in the edge summaries)");
  int A = c.rows * c.cols;
  if (c.edges_per_game <= 0) c.edges_per_game = (c.n_sims + 1) * A;
  if (c.cpuct <= 0.0f) c.cpuct = 1.0f;
  if (c.replay_capacity <= 0) c.replay_capacity = 1;
  if (c.temperature_threshold < 0) c.temperature_threshold = 0;
  if (c.nn_channels <= 0) c.nn_channels = 128;
  if (c.nn_blocks < 0) c.nn_blocks = 10;
  if (c.leaves_per_step < 1) c.leaves_per_step = 1;
  if (c.leaves_per_step > 64) return set_error(YY_ERR_INVALID, "leaves_per_step must be <= 64");
  const uint32_t sym = c.mode_flags & (YY_MODE_EVAL_RANDOM_FORM | YY_MODE_EVAL_AVERAGE_FORMS);
  if (sym == (YY_MODE_EVAL_RANDOM_FORM | YY_MODE_EVAL_AVERAGE_FORMS))
    return set_error(YY_ERR_INVALID, "YY_MODE_EVAL_RANDOM_FORM and YY_MODE_EVAL_AVERAGE_FORMS exclude each other");
  if (sym && c.evaluator != YY_EVAL_NN) return set_error(YY_ERR_INVALID, "symmetric evaluation needs the NN evaluator");
  // in-flight simulations each own a node: keep the worst case inside the node arena
  return YY_OK;
}

static void carve(const yy_engine_config& c, Carver& k, EngineDev& d) {
  const int A = c.rows * c.cols, W = words_for_cells(A);
  const size_t G = (size_t)c.n_games, MN = (size_t)c.n_sims + 2, EC = (size_t)c.edges_per_game;
  d.rows = c.rows; d.cols = c.cols; d.A = A; d.W = W; d.n_games = c.n_games; d.n_sims = c.n_sims;
  d.max_nodes = (int)MN; d.edges_cap = (int)EC; d.max_depth = A + 2;
  d.node_black = k.take<uint64_t>(G * MN * W); d.node_white = k.take<uint64_t>(G * MN * W);
  d.node_edge_base = k.take<int32_t>(G * MN); d.node_n_edges = k.take<int16_t>(G * MN);
  d.node_player = k.take<int8_t>(G * MN); d.node_flags = k.take<uint8_t>(G * MN); d.node_value = k.take<float>(G * MN);
  d.edge_N = k.take<int32_t>(G * EC); d.edge_W = k.take<float>(G * EC); d.edge_P = k.take<float>(G * EC);
  d.edge_cmeta = k.take<uint64_t>(G * EC); d.edge_action = k.take<uint8_t>(G * EC);
  d.g_n_nodes = k.take<int32_t>(G); d.g_n_edges = k.take<int32_t>(G); d.g_sims_done = k.take<int32_t>(G);
  d.g_sim_budget = k.take<int32_t>(G);
  d.K = c.leaves_per_step; d.n_slots = c.n_games * c.leaves_per_step;
  const size_t S = (size_t)d.n_slots;
  d.g_npending = k.take<int32_t>(G);
  d.leaf_node = k.take<int32_t>(S); d.leaf_path_len = k.take<int32_t>(S); d.leaf_path = k.take<int32_t>(S * (size_t)d.max_depth);
  d.leaf_black = k.take<uint64_t>(S * W); d.leaf_white = k.take<uint64_t>(S * W); d.leaf_mask = k.take<uint64_t>(S * W);
  d.leaf_code = k.take<int8_t>(S); d.leaf_active = k.take<uint8_t>(S);
  d.eval_prior = k.take<float>(S * A); d.eval_value = k.take<float>(S); d.active_count = k.take<int32_t>(2);
  d.root_black = k.take<uint64_t>(G * W); d.root_white = k.take<uint64_t>(G * W); d.root_player = k.take<int8_t>(G);
  d.noise = k.take<double>(G * A); d.noise_mask = k.take<uint8_t>(G);
  d.sp_black = k.take<uint64_t>(G * W); d.sp_white = k.take<uint64_t>(G * W); d.sp_player = k.take<int8_t>(G);
  d.sp_step = k.take<int32_t>(G); d.sp_passes = k.take<int32_t>(G); d.sp_serial = k.take<int32_t>(G);
  d.sp_new_game = k.take<uint8_t>(G); d.sp_full = k.take<uint8_t>(G); d.sp_next_serial = k.take<int32_t>(1);
  d.sp_phase = k.take<uint8_t>(G); d.sp_moves_left = k.take<int32_t>(G); d.act_list = k.take<int32_t>(G);
  d.game_quota = -1; d.hook_uniform = nullptr; d.hook_noise = nullptr; d.hook_games = 0; d.hook_plies = 0;
  const size_t RC = (size_t)c.replay_capacity;
  d.replay_cap = (int)RC; d.results_cap = (int)(RC + G + 16);
  d.rp_black = k.take<uint64_t>(RC * W); d.rp_white = k.take<uint64_t>(RC * W); d.rp_counts = k.take<uint16_t>(RC * A);
  d.rp_serial = k.take<int32_t>(RC); d.rp_ply = k.take<int16_t>(RC); d.rp_player = k.take<int8_t>(RC);
  d.rp_results = k.take<int8_t>((size_t)d.results_cap);
  d.stats = k.take<Stats>(1);
}

}  // namespace yy

using namespace yy;

struct yy_engine {
  yy_engine_config cfg;
  EngineDev dev;
  NNState nn;
  bool search_open;
  int step_parity;   // which half of the double-buffered pending-leaf counter the last tree step used
  // scratch pointers for caller-supplied noise in yy_search
  const double* user_noise; const uint8_t* user_noise_mask;
};

namespace {

inline unsigned warp_grid(int n_games) { return (unsigned)(((long long)n_games * 32 + kTreeBlock - 1) / kTreeBlock); }
inline unsigned thread_grid(int n, int block) { return (unsigned)((n + block - 1) / block); }

int launch_root(yy_engine* e, cudaStream_t s, bool prepared = false) {
  YY_DISPATCH_NW(e->dev.A, tree_root_kernel<NW><<<warp_grid(e->dev.n_games), kTreeBlock, 0, s>>>(
      e->dev, make_geo<NW>(e->cfg.rows, e->cfg.cols, e->cfg.rule_flags), prepared ? 1 : 0));
  YY_LAUNCH_CHECK();
  e->step_parity = 0;   // root wrote [0] = n_games, [1] = 0; the first step counts into [1]
  return YY_OK;
}
int launch_step(yy_engine* e, cudaStream_t s) {
  e->step_parity ^= 1;
  YY_DISPATCH_NW(e->dev.A, tree_step_kernel<NW><<<warp_grid(e->dev.n_games), kTreeBlock, 0, s>>>(
      e->dev, make_geo<NW>(e->cfg.rows, e->cfg.cols, e->cfg.rule_flags), e->step_parity));
  YY_LAUNCH_CHECK();
  return YY_OK;
}
// the form every network evaluation of the engine uses (mode_flags)
FormSpec engine_forms(const yy_engine* e) {
  FormSpec f;
  if (e->cfg.mode_flags & YY_MODE_EVAL_RANDOM_FORM) { f.mode = YY_FORM_HASHED; f.seed = e->cfg.seed; }
  if (e->cfg.mode_flags & YY_MODE_EVAL_AVERAGE_FORMS) f.mode = YY_FORM_AVERAGE;
  return f;
}
// network forward = the persistent kernel with one iteration and no tree step (in chunks that fit the head-feature scratch)
int engine_forward(yy_engine* e, const uint64_t* black, const uint64_t* white, int64_t count, float* policy, float* value,
                   float* logits, const FormSpec& forms, cudaStream_t s) {
  const int E = form_entries(forms.mode, e->cfg.rows, e->cfg.cols);
  int64_t chunk = e->nn.max_entries / E < e->nn.max_boards ? e->nn.max_entries / E : e->nn.max_boards;
  if (chunk < 1)
    return set_error(YY_ERR_INVALID, "averaging over %d forms needs a head-feature scratch of >= %d boards (n_games x leaves_per_step), "
                     "or an engine created with YY_MODE_EVAL_AVERAGE_FORMS", E, E);
  for (int64_t done = 0; done < count; done += chunk) {
    const int64_t n = (count - done) < chunk ? (count - done) : chunk;
    int rc = nn_fused_run(e->nn, nullptr, e->cfg.rule_flags, black + done * e->dev.W, white + done * e->dev.W, n, policy + done * e->dev.A,
                          value + done, logits ? logits + done * e->dev.A : nullptr, 1, true, YY_FUSED_FORWARD, forms, s);
    if (rc) return rc;
  }
  return YY_OK;
}
// evaluator on the pending leaf batch (STUB is fused into the tree kernels)
int run_evaluator(yy_engine* e, cudaStream_t s) {
  if (e->cfg.evaluator == YY_EVAL_STUB) return YY_OK;
  if (e->cfg.evaluator == YY_EVAL_NN)
    return engine_forward(e, e->dev.leaf_black, e->dev.leaf_white, e->dev.n_slots, e->dev.eval_prior, e->dev.eval_value, nullptr,
                          engine_forms(e), s);
  return set_error(YY_ERR_STATE, "external evaluator: use yy_search_begin / yy_search_advance");
}
// full search over the roots already stored in dev.root_* (noise pointers already set in dev); `prepared`: the
// lock-step self-play driver's search, with the simulation budget sp_prepare_kernel chose per game
int search_core(yy_engine* e, cudaStream_t s, bool prepared = false) {
  int rc = launch_root(e, s, prepared); if (rc) return rc;
  if (e->cfg.leaves_per_step <= 1 && !(e->cfg.mode_flags & YY_MODE_STEP_KERNELS) && e->cfg.evaluator != YY_EVAL_EXTERNAL) {
    // the whole search in ONE persistent kernel: every CTA owns a run of games from the first to the last simulation
    // (the launch ends as soon as no game has work left; a game advances by at least one simulation every two steps)
    return nn_fused_run(e->nn, &e->dev, e->cfg.rule_flags, e->dev.leaf_black, e->dev.leaf_white, e->dev.n_slots, e->dev.eval_prior,
                        e->dev.eval_value, nullptr, 2 * (e->cfg.n_sims + 1), e->cfg.evaluator == YY_EVAL_NN, YY_FUSED_SEARCH,
                        engine_forms(e), s);
  }
  if (e->cfg.leaves_per_step <= 1) {      // deterministic mode: exactly n_sims + 1 lock-steps, no host synchronisation
    for (int i = 0; i <= e->cfg.n_sims; ++i) {
      rc = run_evaluator(e, s); if (rc) return rc;
      rc = launch_step(e, s); if (rc) return rc;
    }
    return YY_OK;
  }
  // throughput mode: a step retires up to K simulations per game; poll the pending-leaf counter every few steps
  for (int i = 0; i <= e->cfg.n_sims; ++i) {
    rc = run_evaluator(e, s); if (rc) return rc;
    rc = launch_step(e, s); if (rc) return rc;
    if ((i & 3) == 3 || i == e->cfg.n_sims) {
      int32_t active = 0;
      YY_CUDA_OK(cudaMemcpyAsync(&active, e->dev.active_count + e->step_parity, 4, cudaMemcpyDeviceToHost, s));
      YY_CUDA_OK(cudaStreamSynchronize(s));
      if (active == 0) break;
    }
  }
  return YY_OK;
}
int copy_roots(yy_engine* e, const uint64_t* rb, const uint64_t* rw, const int8_t* rp, const double* noise,
               const uint8_t* noise_mask, cudaStream_t s) {
  const size_t G = (size_t)e->dev.n_games, W = (size_t)e->dev.W, A = (size_t)e->dev.A;
  if (!rb || !rw || !rp) return set_error(YY_ERR_INVALID, "null root pointer");
  YY_CUDA_OK(cudaMemcpyAsync(e->dev.root_black, rb, G * W * 8, cudaMemcpyDeviceToDevice, s));
  YY_CUDA_OK(cudaMemcpyAsync(e->dev.root_white, rw, G * W * 8, cudaMemcpyDeviceToDevice, s));
  YY_CUDA_OK(cudaMemcpyAsync(e->dev.root_player, rp, G, cudaMemcpyDeviceToDevice, s));
  if (noise && noise_mask) {
    YY_CUDA_OK(cudaMemcpyAsync(e->dev.noise, noise, G * A * 8, cudaMemcpyDeviceToDevice, s));
    YY_CUDA_OK(cudaMemcpyAsync(e->dev.noise_mask, noise_mask, G, cudaMemcpyDeviceToDevice, s));
  } else {
    YY_CUDA_OK(cudaMemsetAsync(e->dev.noise_mask, 0, G, s));
  }
  return YY_OK;
}

}  // namespace

extern "C" {

int64_t yy_engine_workspace_bytes(const yy_engine_config* cfg) {
  if (!cfg) { set_error(YY_ERR_INVALID, "null config"); return YY_ERR_INVALID; }
  yy_engine_config c = *cfg;
  int rc = normalise_cfg(c); if (rc) return rc;
  Carver k{nullptr, 0}; EngineDev d{};
  carve(c, k, d);
  size_t total = ((k.off + 255) & ~(size_t)255) + nn_workspace_bytes(c);
  return (int64_t)total;
}

yy_engine* yy_engine_create(const yy_engine_config* cfg, void* workspace, int64_t workspace_bytes) {
  if (!cfg || !workspace) { set_error(YY_ERR_INVALID, "null config/workspace"); return nullptr; }
  yy_engine_config c = *cfg;
  if (normalise_cfg(c)) return nullptr;
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd == 0) { cudaGetLastError(); set_error(YY_ERR_NO_DEVICE, "no CUDA device: the engine has no CPU fallback"); return nullptr; }
  if (cudaSetDevice(c.device) != cudaSuccess) { set_error(YY_ERR_CUDA, "cudaSetDevice(%d) failed", c.device); return nullptr; }
  int64_t need = yy_engine_workspace_bytes(&c);
  if (workspace_bytes < need) { set_error(YY_ERR_INVALID, "workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)need); return nullptr; }
  if (((uintptr_t)workspace & 255) != 0) { set_error(YY_ERR_INVALID, "workspace must be 256-byte aligned"); return nullptr; }
  yy_engine* e = new (std::nothrow) yy_engine();
  if (!e) { set_error(YY_ERR_INVALID, "out of host memory"); return nullptr; }
  e->cfg = c; e->search_open = false; e->step_parity = 0; e->user_noise = nullptr; e->user_noise_mask = nullptr;
  Carver k{(char*)workspace, 0};
  carve(c, k, e->dev);
  e->dev.cpuct = c.cpuct; e->dev.eps = (double)c.dirichlet_epsilon; e->dev.alpha = (double)c.dirichlet_alpha;
  e->dev.keep_f32 = (float)(1.0 - (double)c.dirichlet_epsilon);
  e->dev.evaluator = c.evaluator; e->dev.mode_flags = c.mode_flags; e->dev.temperature_threshold = c.temperature_threshold;
  e->dev.seed = c.seed;
  e->dev.cap_threshold = 1ull << 32; e->dev.fast_sims = c.n_sims;      // playout cap off: every move a full search
  e->dev.max_descents = c.descents_per_step == 0 ? 4 : (c.descents_per_step < 0 ? 0 : c.descents_per_step);
  size_t off = (k.off + 255) & ~(size_t)255;
  if (nn_init(e->nn, c, (char*)workspace + off) != YY_OK) { delete e; return nullptr; }
  sp_reset_kernel<<<thread_grid(c.n_games, 128), 128>>>(e->dev);
  count_launch();
  if (cudaDeviceSynchronize() != cudaSuccess) { set_error(YY_ERR_CUDA, "engine init: %s", cudaGetErrorString(cudaGetLastError())); delete e; return nullptr; }
  return e;
}

void yy_engine_destroy(yy_engine* e) { if (e) { nn_destroy(e->nn); delete e; } }

int64_t yy_nn_weight_bytes(int rows, int cols, int channels, int blocks) { return nn_weight_bytes(rows, cols, channels, blocks); }
int yy_engine_load_weights(yy_engine* e, const void* weights, int64_t bytes) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  return nn_load_weights(e->nn, weights, bytes);
}

int yy_search(yy_engine* e, const uint64_t* rb, const uint64_t* rw, const int8_t* rp, const double* noise,
              const uint8_t* noise_mask, int32_t* out_counts, void* stream) {
  if (!e || !out_counts) return set_error(YY_ERR_INVALID, "null argument");
  if (e->cfg.evaluator == YY_EVAL_EXTERNAL) return set_error(YY_ERR_STATE, "external evaluator: use yy_search_begin / yy_search_advance");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = copy_roots(e, rb, rw, rp, noise, noise_mask, s); if (rc) return rc;
  rc = search_core(e, s); if (rc) return rc;
  tree_counts_kernel<<<thread_grid(e->dev.n_games, 128), 128, 0, s>>>(e->dev, out_counts, nullptr);
  YY_LAUNCH_CHECK();
  return YY_OK;
}

int yy_search_begin(yy_engine* e, const uint64_t* rb, const uint64_t* rw, const int8_t* rp, const double* noise,
                    const uint8_t* noise_mask, void* stream) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = copy_roots(e, rb, rw, rp, noise, noise_mask, s); if (rc) return rc;
  rc = launch_root(e, s); if (rc) return rc;
  e->search_open = true;
  return YY_OK;
}

int yy_search_advance(yy_engine* e, const float* priors, const float* values, int32_t* out_active, void* stream) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  if (!e->search_open) return set_error(YY_ERR_STATE, "yy_search_advance without yy_search_begin");
  cudaStream_t s = (cudaStream_t)stream;
  const size_t G = (size_t)e->dev.n_slots, A = (size_t)e->dev.A;
  if (priors && values) {
    YY_CUDA_OK(cudaMemcpyAsync(e->dev.eval_prior, priors, G * A * 4, cudaMemcpyDeviceToDevice, s));
    YY_CUDA_OK(cudaMemcpyAsync(e->dev.eval_value, values, G * 4, cudaMemcpyDeviceToDevice, s));
  } else if (e->cfg.evaluator != YY_EVAL_STUB) {
    int rc = run_evaluator(e, s); if (rc) return rc;
  }
  int rc = launch_step(e, s); if (rc) return rc;
  if (out_active) {
    YY_CUDA_OK(cudaMemcpyAsync(out_active, e->dev.active_count + e->step_parity, 4, cudaMemcpyDeviceToHost, s));
    YY_CUDA_OK(cudaStreamSynchronize(s));
    if (*out_active == 0) e->search_open = false;
  }
  return YY_OK;
}

int yy_search_counts(yy_engine* e, int32_t* out_counts, float* out_child_w, void* stream) {
  if (!e || !out_counts) return set_error(YY_ERR_INVALID, "null argument");
  tree_counts_kernel<<<thread_grid(e->dev.n_games, 128), 128, 0, (cudaStream_t)stream>>>(e->dev, out_counts, out_child_w);
  YY_LAUNCH_CHECK();
  return YY_OK;
}

int yy_engine_tree_view(yy_engine* e, yy_tree_view* out) {
  if (!e || !out) return set_error(YY_ERR_INVALID, "null argument");
  const EngineDev& d = e->dev;
  out->max_nodes = d.max_nodes; out->edges_cap = d.edges_cap; out->W = d.W;
  out->n_nodes = d.g_n_nodes; out->n_edges_used = d.g_n_edges;
  out->node_black = d.node_black; out->node_white = d.node_white;
  out->node_edge_base = d.node_edge_base; out->node_n_edges = d.node_n_edges; out->node_player = d.node_player;
  out->node_flags = d.node_flags; out->node_value = d.node_value;
  out->edge_N = d.edge_N; out->edge_W = d.edge_W; out->edge_P = d.edge_P; out->edge_child_meta = d.edge_cmeta; out->edge_action = d.edge_action;
  return YY_OK;
}

const uint64_t* yy_engine_leaf_black(yy_engine* e) { return e ? e->dev.leaf_black : nullptr; }
const uint64_t* yy_engine_leaf_white(yy_engine* e) { return e ? e->dev.leaf_white : nullptr; }
const uint8_t* yy_engine_leaf_active(yy_engine* e) { return e ? e->dev.leaf_active : nullptr; }
const uint64_t* yy_engine_game_black(yy_engine* e) { return e ? e->dev.sp_black : nullptr; }
const uint64_t* yy_engine_game_white(yy_engine* e) { return e ? e->dev.sp_white : nullptr; }
const int8_t* yy_engine_game_player(yy_engine* e) { return e ? e->dev.sp_player : nullptr; }

int yy_evaluate(yy_engine* e, const uint64_t* black, const uint64_t* white, int64_t count, float* out_policy,
                float* out_value, float* out_logits, void* stream) {
  if (!e || !black || !white || !out_policy || !out_value) return set_error(YY_ERR_INVALID, "null argument");
  if (count <= 0) return YY_OK;
  cudaStream_t s = (cudaStream_t)stream;
  if (e->cfg.evaluator == YY_EVAL_NN) return engine_forward(e, black, white, count, out_policy, out_value, out_logits, engine_forms(e), s);
  if (e->cfg.evaluator == YY_EVAL_STUB) {
    YY_DISPATCH_NW(e->dev.A, stub_eval_kernel<NW><<<thread_grid((int)count, 128), 128, 0, s>>>(
        make_geo<NW>(e->cfg.rows, e->cfg.cols, e->cfg.rule_flags), e->dev.W, black, white, count, out_policy, out_value));
    YY_LAUNCH_CHECK();
    return YY_OK;
  }
  return set_error(YY_ERR_STATE, "yy_evaluate needs the STUB or NN evaluator");
}

int yy_evaluate_form(yy_engine* e, const uint64_t* black, const uint64_t* white, int64_t count, int32_t form, float* out_policy,
                     float* out_value, float* out_logits, void* stream) {
  if (!e || !black || !white || !out_policy || !out_value) return set_error(YY_ERR_INVALID, "null argument");
  if (e->cfg.evaluator != YY_EVAL_NN) return set_error(YY_ERR_INVALID, "yy_evaluate_form needs the NN evaluator");
  FormSpec f;
  if (form == -1) f.mode = YY_FORM_AVERAGE;
  else if (form_valid(form, e->cfg.rows, e->cfg.cols)) { f.mode = YY_FORM_FIXED; f.form = form; }
  else return set_error(YY_ERR_INVALID, "form %d is not a form of a %dx%d board (0..7 square, 0/2/4/5 rectangular; -1 = average)",
                        form, e->cfg.rows, e->cfg.cols);
  if (f.mode == YY_FORM_AVERAGE && out_logits) return set_error(YY_ERR_INVALID, "no logits when averaging over the forms");
  if (count <= 0) return YY_OK;
  return engine_forward(e, black, white, count, out_policy, out_value, out_logits, f, (cudaStream_t)stream);
}

int yy_engine_set_profiling(yy_engine* e, int enable) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  return nn_set_profiling(e->nn, enable);
}
// developer tool: per-layer clock64 stamps of the tower kernel's CTA 0 / first group into dbg_dev (>= 4*(2*blocks+2) int64)
int yy_engine_set_debug_stamps(yy_engine* e, long long* dbg_dev) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  e->nn.dbg = dbg_dev;
  return YY_OK;
}
int yy_engine_set_debug_flags(yy_engine* e, int flags) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  e->nn.dbg_flags = flags;
  return YY_OK;
}
int yy_engine_get_profile(yy_engine* e, int64_t* tower_launches, double* tower_ms, int64_t* tower_boards) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  long long l = 0, b = 0; double ms = 0.0;
  int rc = nn_get_profile(e->nn, &l, &ms, &b); if (rc) return rc;
  if (tower_launches) *tower_launches = l;
  if (tower_ms) *tower_ms = ms;
  if (tower_boards) *tower_boards = b;
  return YY_OK;
}

int yy_selfplay_reset(yy_engine* e, void* stream) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  sp_reset_kernel<<<thread_grid(e->dev.n_games, 128), 128, 0, (cudaStream_t)stream>>>(e->dev);
  YY_LAUNCH_CHECK();
  return YY_OK;
}

// the persistent kernel plays the games itself unless the search has to run as per-step kernels
static bool rolling_capable(const yy_engine* e) {
  return e->cfg.leaves_per_step <= 1 && !(e->cfg.mode_flags & YY_MODE_STEP_KERNELS) && e->cfg.evaluator != YY_EVAL_EXTERNAL;
}
static int launch_rolling(yy_engine* e, int moves_per_slot, long long iterations, cudaStream_t s) {
  sp_budget_kernel<<<thread_grid(e->dev.n_games, 128), 128, 0, s>>>(e->dev, moves_per_slot);
  YY_LAUNCH_CHECK();
  if (iterations > 0x7fffffffll) iterations = 0x7fffffffll;
  return nn_fused_run(e->nn, &e->dev, e->cfg.rule_flags, e->dev.leaf_black, e->dev.leaf_white, e->dev.n_slots, e->dev.eval_prior,
                      e->dev.eval_value, nullptr, (int)iterations, e->cfg.evaluator == YY_EVAL_NN, YY_FUSED_SELFPLAY,
                      engine_forms(e), s);
}

int yy_selfplay_run(yy_engine* e, int32_t n_moves, void* stream) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  if (e->cfg.evaluator == YY_EVAL_EXTERNAL) return set_error(YY_ERR_STATE, "self-play needs the STUB or NN evaluator");
  cudaStream_t s = (cudaStream_t)stream;
  if (n_moves <= 0) return YY_OK;
  // ONE launch: every slot makes n_moves moves at its own pace (a search needs at most 2 (n_sims + 1) steps, usually
  // n_sims + 1 or fewer); the launch ends when the last slot has made its moves
  if (rolling_capable(e)) return launch_rolling(e, n_moves, 2ll * n_moves * (e->cfg.n_sims + 1), s);
  if (e->dev.game_quota >= 0) return set_error(YY_ERR_STATE, "a game quota needs the persistent kernel (leaves_per_step 1, no YY_MODE_STEP_KERNELS)");
  const unsigned grid = thread_grid(e->dev.n_games, 128);
  for (int mv = 0; mv < n_moves; ++mv) {
    YY_DISPATCH_NW(e->dev.A, sp_prepare_kernel<NW><<<grid, 128, 0, s>>>(e->dev, make_geo<NW>(e->cfg.rows, e->cfg.cols, e->cfg.rule_flags)));
    YY_LAUNCH_CHECK();
    YY_DISPATCH_NW(e->dev.A, sp_noise_kernel<NW><<<grid, 128, 0, s>>>(e->dev, make_geo<NW>(e->cfg.rows, e->cfg.cols, e->cfg.rule_flags)));
    YY_LAUNCH_CHECK();
    int rc = search_core(e, s, true); if (rc) return rc;
    YY_DISPATCH_NW(e->dev.A, sp_move_kernel<NW><<<grid, 128, 0, s>>>(e->dev, make_geo<NW>(e->cfg.rows, e->cfg.cols, e->cfg.rule_flags)));
    YY_LAUNCH_CHECK();
  }
  return YY_OK;
}

int yy_selfplay_advance(yy_engine* e, int64_t iterations, void* stream) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  if (!rolling_capable(e)) return set_error(YY_ERR_STATE, "yy_selfplay_advance needs the persistent kernel (STUB or NN evaluator, leaves_per_step 1)");
  if (iterations <= 0) return YY_OK;
  return launch_rolling(e, kMovesUnlimited, iterations, (cudaStream_t)stream);
}

int yy_selfplay_set_quota(yy_engine* e, int64_t total_games) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  e->dev.game_quota = total_games < 0 ? -1 : (long long)total_games;
  return YY_OK;
}

int yy_selfplay_set_playout_cap(yy_engine* e, double full_prob, int32_t fast_sims) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  if (e->cfg.evaluator == YY_EVAL_EXTERNAL) return set_error(YY_ERR_STATE, "self-play needs the STUB or NN evaluator");
  if (!(full_prob >= 0.0 && full_prob <= 1.0)) return set_error(YY_ERR_INVALID, "full_prob must be in [0, 1]");
  if (fast_sims < 1 || fast_sims > e->cfg.n_sims)
    return set_error(YY_ERR_INVALID, "fast_sims must be in [1, n_sims = %d], not %d", e->cfg.n_sims, (int)fast_sims);
  e->dev.cap_threshold = (uint64_t)llround(full_prob * 4294967296.0);
  e->dev.fast_sims = fast_sims;
  return YY_OK;
}

int yy_selfplay_set_random_stream(yy_engine* e, const double* uniforms_dev, const double* noise_dev, int32_t n_games, int32_t n_plies) {
  if (!e) return set_error(YY_ERR_INVALID, "null engine");
  if ((uniforms_dev || noise_dev) && (n_games <= 0 || n_plies <= 0)) return set_error(YY_ERR_INVALID, "recorded stream needs n_games, n_plies > 0");
  e->dev.hook_uniform = uniforms_dev; e->dev.hook_noise = noise_dev; e->dev.hook_games = n_games; e->dev.hook_plies = n_plies;
  return YY_OK;
}

int yy_selfplay_get_stats(yy_engine* e, yy_selfplay_stats* out, void* stream) {
  if (!e || !out) return set_error(YY_ERR_INVALID, "null argument");
  Stats h;
  YY_CUDA_OK(cudaMemcpyAsync(&h, e->dev.stats, sizeof(Stats), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  YY_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
  out->moves = (int64_t)h.moves; out->evals = (int64_t)h.evals; out->games_finished = (int64_t)h.games_finished;
  out->examples = (int64_t)h.examples; out->sims = (int64_t)h.sims; out->overflow = h.overflow; out->max_depth = h.max_depth;
  out->tower_evals = (int64_t)h.tower_evals;
  if (h.overflow) return set_error(YY_ERR_CAPACITY, "a tree arena overflowed: raise edges_per_game");
  return YY_OK;
}

const void* yy_selfplay_stats_dev(yy_engine* e) { return e ? (const void*)e->dev.stats : nullptr; }

int yy_selfplay_replay(yy_engine* e, yy_replay_view* out) {
  if (!e || !out) return set_error(YY_ERR_INVALID, "null argument");
  out->black = e->dev.rp_black; out->white = e->dev.rp_white; out->counts = e->dev.rp_counts;
  out->game_serial = e->dev.rp_serial; out->ply = e->dev.rp_ply; out->player = e->dev.rp_player;
  out->results = e->dev.rp_results; out->results_capacity = e->dev.results_cap;
  return YY_OK;
}

}  // extern "C"
