// yy_engine.cuh -- device-side view of the engine state (HBM-resident MCTS forest + self-play slots).
//
// One tree per game, all arrays struct-of-arrays and game-major so that the warp that owns a game
// reads its children's (N, W, P) with coalesced 128-byte requests:
//   node arrays  [n_games][max_nodes]   state bitboards, player, flags, edge range, cached value
//   edge arrays  [n_games][edges_cap]   one slot per (node, legal action) in ascending action order:
//                                       N int32, W float32, P float32, child int32, action uint8
// A reference Node (src/yin_yang/ai/mcts.py:28-48) is split in two: its statistics (visits, value_sum,
// prior, action) live in the parent's edge slot, its state (board, player, is_terminal, terminal_value,
// children) in a node record created when the simulation that first reaches it expands it.
#pragma once
#include "yy_common.cuh"

namespace yy {

enum : uint8_t { NODE_EXPANDED = 1, NODE_TERMINAL = 2, NODE_NOCHILD = 4 };

struct Stats {  // device counters (unsigned long long for atomicAdd)
  unsigned long long moves, evals, games_finished, examples, sims;
  int overflow, max_depth;
  unsigned long long tower_evals;   // boards the persistent kernel evaluated (every one of them a pending leaf)
};

struct EngineDev {
  // geometry / config
  int rows, cols, A, W;
  int n_games, n_sims, max_nodes, edges_cap, max_depth;
  int max_descents; // persistent kernel: simulations a game may start per step (0 = until a leaf needs an evaluation)
  int K, n_slots;   // leaves per game per step (1 = deterministic mode), evaluation slots = n_games * K
  float cpuct;
  float keep_f32;   // f32(1 - eps)            (mcts.py:309-311 under numpy>=2)
  double eps;       // dirichlet epsilon
  double alpha;
  int evaluator;
  uint32_t mode_flags;
  int temperature_threshold;
  uint64_t seed;
  // playout cap randomisation of self-play (yy_selfplay_set_playout_cap): a move is a full search iff
  // hash(seed, serial, ply) >> 32 < cap_threshold (2^32 = always: the default), otherwise a fast one of fast_sims
  uint64_t cap_threshold;
  int fast_sims;
  // nodes
  uint64_t* node_black; uint64_t* node_white;
  int32_t* node_edge_base; int16_t* node_n_edges; int8_t* node_player; uint8_t* node_flags; float* node_value;
  // edges
  int32_t* edge_N; float* edge_W; float* edge_P; uint64_t* edge_cmeta; uint8_t* edge_action;
  // per game search state
  int32_t* g_n_nodes; int32_t* g_n_edges; int32_t* g_sims_done;
  int32_t* g_sim_budget; // simulations the game's current search runs (n_sims, or fast_sims for a fast self-play move)
  int32_t* g_npending;   // leaves waiting for the evaluator; 0 = no search in progress; -1 = search in progress, no leaf this step
  // pending leaf batch (evaluator input), slot = game*K + k: node id, recorded path, state, rules result
  int32_t* leaf_node; int32_t* leaf_path_len; int32_t* leaf_path;
  uint64_t* leaf_black; uint64_t* leaf_white; uint64_t* leaf_mask; int8_t* leaf_code; uint8_t* leaf_active;
  float* eval_prior;  // [n_slots][A] raw softmax entries (mcts.py:77-78: unmasked, un-normalised)
  float* eval_value;  // [n_slots]
  int32_t* active_count;
  // root inputs for the current search
  uint64_t* root_black; uint64_t* root_white; int8_t* root_player;
  double* noise; uint8_t* noise_mask;
  // self-play slots
  uint64_t* sp_black; uint64_t* sp_white; int8_t* sp_player; int32_t* sp_step; int32_t* sp_passes; int32_t* sp_serial;
  uint8_t* sp_new_game;
  uint8_t* sp_full;         // 1 = the slot's current search is a full one: its move is recorded in the replay ring
  int32_t* sp_next_serial;
  // rolling self-play inside the persistent kernel (yy_fused.cu): a slot whose search is complete makes its move and
  // roots the next search at once, independently of the other slots
  uint8_t* sp_phase;        // 1 = the slot's tree belongs to a self-play search in progress / just completed
  int32_t* sp_moves_left;   // moves the slot may still make in this launch (INT_MAX = unlimited)
  long long game_quota;     // games that may be started in total since the last reset; < 0 = unlimited
  int32_t* act_list;        // [n_games] per CTA run: the games with a pending leaf, compacted, for the current iteration
  // arena (yy_arena_run): n_games = 2G slots, slot j searches for model A and slot G + j for model B in arena game j.
  // Game j keeps its board, player to move and ply in self-play slot j (sp_black, sp_white, sp_player, sp_step); sp_phase[s]
  // = 1 while slot s has a search of the game in progress.
  int32_t* ar_turn;         // [G] slot whose model is to move in game j, -1 once the game is over (the hand-off flag)
  int8_t* ar_code;          // [G] YY_RESULT_* after the last move (player to move's view), 0 if the ply cap ended the game
  uint8_t* ar_a_black;      // [G] 1 = model A plays black in game j
  int ar_max_plies;         // a game that reaches this many plies ends with code 0
  // recorded random stream (test seam; replaces the np.random.choice / np.random.dirichlet draws of self_play.py:143-160
  // and mcts.py:303-306): uniforms [hook_games][hook_plies], Dirichlet samples [hook_games][A]; nullptr = Philox
  const double* hook_uniform; const double* hook_noise; int hook_games, hook_plies;
  // replay ring
  int replay_cap; int results_cap;
  uint64_t* rp_black; uint64_t* rp_white; uint16_t* rp_counts; int32_t* rp_serial; int16_t* rp_ply; int8_t* rp_player;
  int8_t* rp_results;
  Stats* stats;
};

}  // namespace yy
