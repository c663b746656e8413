// yy_selfplay_dev.cuh -- device-side episode driver of ONE game: SelfPlayWorker.play_game (src/yin_yang/ai/self_play.py:72-192)
// cut at the points where it calls MCTS.search.  The *_one functions are single-thread code (one thread per game in the
// lock-step kernels of yy_tree.cu, lane 0 of the game's warp inside the persistent kernel of yy_fused.cu);
// tree_root_game and sp_advance_game are executed by the whole warp that owns the game.
#pragma once
#include "yy_tree_dev.cuh"

namespace yy {

constexpr int kMovesUnlimited = 0x7fffffff;

__device__ __forceinline__ void finish_game(const EngineDev& e, int gi, int code) {
  int serial = e.sp_serial[gi];
  if (serial >= 0) e.rp_results[serial % e.results_cap] = (int8_t)code;
  atomicAdd(&e.stats->games_finished, 1ull);
  e.sp_new_game[gi] = 1;
}

// Serial number of the next game (a dense sequence: game s of a run is the same game whichever slot plays it -- every
// random draw is keyed by (seed, s, ply)); -1 when the quota of games is used up.
__device__ __forceinline__ int next_game_serial(const EngineDev& e) {
  const int s = atomicAdd(e.sp_next_serial, 1);
  if (e.game_quota >= 0 && (long long)s >= e.game_quota) { atomicSub(e.sp_next_serial, 1); return -1; }
  return s;
}

// Top of the play_game loop (self_play.py:91-125): new game if needed, pass / double-pass handling, then the root of
// the next search.  search player = 1 always under YY_MODE_SEARCH_AS_BLACK (self_play.py:99,135-137).
// Playout cap: the search is a full one (n_sims, noise at ply 0, recorded) or a fast one (fast_sims, no noise, not
// recorded) as playout_full decides for (seed, serial, ply).
// Returns the simulation budget of the search, or -1 when the slot needs a new game and the quota is used up (the slot
// idles).
template <int NW>
__device__ __forceinline__ int sp_prepare_one(const EngineDev& e, const Geo<NW>& g, int gi) {
  BB<NW> b = load_bb<NW>(e.sp_black, gi, e.W), w = load_bb<NW>(e.sp_white, gi, e.W);
  int player = e.sp_player[gi], step = e.sp_step[gi], passes = e.sp_passes[gi];
  int sp = 1;
  for (;;) {
    if (e.sp_new_game[gi]) {
      const int serial = next_game_serial(e);
      if (serial < 0) { e.sp_serial[gi] = -1; return -1; }
      b = bb_zero<NW>(); w = bb_zero<NW>(); player = 1; step = 0; passes = 0;
      e.sp_serial[gi] = serial;
      e.sp_new_game[gi] = 0;
      e.rp_results[serial % e.results_cap] = 0;           // the slot may hold the result of game serial - results_cap
    }
    sp = (e.mode_flags & YY_MODE_SEARCH_AS_BLACK) ? 1 : player;
    if (any(legal_for(g, b, w, sp))) { passes = 0; break; }
    ++passes;                                             // self_play.py:103-106
    if (passes >= 2) {                                    // self_play.py:108-121
      int code = ended_code(g, b, w, player);
      if (code == 0) code = YY_RESULT_DRAW;
      finish_game(e, gi, code);
      continue;
    }
    player = -player;                                     // self_play.py:124-125
  }
  store_bb<NW>(e.sp_black, gi, e.W, b); store_bb<NW>(e.sp_white, gi, e.W, w);
  e.sp_player[gi] = (int8_t)player; e.sp_step[gi] = step; e.sp_passes[gi] = passes;
  store_bb<NW>(e.root_black, gi, e.W, b); store_bb<NW>(e.root_white, gi, e.W, w);
  e.root_player[gi] = (int8_t)sp;
  const bool full = playout_full(e.seed, e.sp_serial[gi], step, e.cap_threshold);
  e.sp_full[gi] = full ? 1 : 0;
  e.noise_mask[gi] = (full && step == 0 && e.eps > 0.0) ? 1 : 0;  // add_noise = (step == 0), self_play.py:131
  return full ? e.n_sims : e.fast_sims;
}

__device__ inline double gamma_sample(Philox& rng, double a) {
  // Marsaglia-Tsang; for a < 1: G(a) = G(a+1) * U^(1/a)
  double boost = 1.0;
  if (a < 1.0) { boost = pow(rng.uniform(), 1.0 / a); a += 1.0; }
  const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
  for (;;) {
    double u1 = rng.uniform(), u2 = rng.uniform();
    double x = sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
    double v = 1.0 + c * x;
    if (v <= 0.0) continue;
    v = v * v * v;
    double u = rng.uniform();
    if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) return boost * d * v;
  }
}

// np.random.dirichlet([alpha]*k) for the legal root actions of a game at step 0 (mcts.py:303-306)
template <int NW>
__device__ __forceinline__ void sp_noise_one(const EngineDev& e, const Geo<NW>& g, int gi) {
  if (!e.noise_mask[gi]) return;
  BB<NW> b = load_bb<NW>(e.root_black, gi, e.W), w = load_bb<NW>(e.root_white, gi, e.W);
  const int k = popcount(legal_for(g, b, w, e.root_player[gi]));
  const int serial = e.sp_serial[gi];
  double* out = e.noise + (long long)gi * e.A;
  if (e.hook_noise && serial >= 0 && serial < e.hook_games) {      // recorded sample (already normalised)
    const double* src = e.hook_noise + (long long)serial * e.A;
    for (int i = 0; i < k; ++i) out[i] = src[i];
    return;
  }
  Philox rng(e.seed, (uint64_t)(uint32_t)serial, 0x6e6f697365ull);
  double sum = 0.0;
  for (int i = 0; i < k; ++i) { double x = gamma_sample(rng, e.alpha); out[i] = x; sum += x; }
  if (sum <= 0.0) { for (int i = 0; i < k; ++i) out[i] = 1.0 / k; }
  else { for (int i = 0; i < k; ++i) out[i] /= sum; }
}

// After the search (self_play.py:139-190): store the example, pick the action (temperature 1 for the first
// `temperature_threshold` moves -- np.random.choice(A, p = pi): the first action whose cumulative probability exceeds a
// uniform draw -- then a uniform choice among the most visited, np.random.choice(best_moves)), apply it with the REAL
// player (illegal -> silently dropped, yin_yang_logic.py:24-29), test for the end of the game.
template <int NW>
__device__ __forceinline__ void sp_move_one(const EngineDev& e, const Geo<NW>& g, int gi) {
  const long long nb = (long long)gi * e.max_nodes, eb = (long long)gi * e.edges_cap;
  BB<NW> b = load_bb<NW>(e.sp_black, gi, e.W), w = load_bb<NW>(e.sp_white, gi, e.W);
  int player = e.sp_player[gi], step = e.sp_step[gi];
  const int serial = e.sp_serial[gi];
  const int base = e.node_edge_base[nb], cnt = (e.node_flags[nb] & NODE_EXPANDED) ? e.node_n_edges[nb] : 0;
  // example record (board before the move, visit counts; pi = counts/sum on the host in float64) -- full searches only:
  // a fast search of the playout cap only advances the game
  uint16_t* rc = nullptr;
  if (e.sp_full[gi]) {
    unsigned long long slot64 = atomicAdd(&e.stats->examples, 1ull);
    long long slot = (long long)(slot64 % (unsigned long long)e.replay_cap);
    store_bb<NW>(e.rp_black, slot, e.W, b); store_bb<NW>(e.rp_white, slot, e.W, w);
    rc = e.rp_counts + slot * e.A;
    for (int a = 0; a < e.A; ++a) rc[a] = 0;
    e.rp_serial[slot] = serial; e.rp_ply[slot] = (int16_t)step; e.rp_player[slot] = (int8_t)player;
  }
  long long total = 0; int maxn = -1, nmax = 0;
  for (int k = 0; k < cnt; ++k) {
    int n = e.edge_N[eb + base + k];
    if (rc) rc[e.edge_action[eb + base + k]] = (uint16_t)(n > 65535 ? 65535 : n);
    total += n;
    if (n > maxn) { maxn = n; nmax = 1; } else if (n == maxn) ++nmax;
  }
  // one uniform draw per move: the recorded stream when there is one, else Philox keyed by (seed, game, ply)
  double u;
  if (e.hook_uniform && serial >= 0 && serial < e.hook_games && step < e.hook_plies) u = e.hook_uniform[(long long)serial * e.hook_plies + step];
  else { Philox rng(e.seed, (uint64_t)(uint32_t)serial, 0x1000ull + (uint64_t)step); u = rng.uniform(); }
  int action = -1;
  if (cnt > 0) {
    if (step < e.temperature_threshold && total > 0) {       // temperature 1: sample proportional to visits
      long long r = (long long)(u * (double)total);
      if (r >= total) r = total - 1;
      long long acc = 0;
      for (int k = 0; k < cnt; ++k) { acc += e.edge_N[eb + base + k]; if (r < acc) { action = e.edge_action[eb + base + k]; break; } }
    } else if (total > 0) {                                    // temperature 0: uniform choice among the maxima
      int pick = (int)(u * (double)nmax);
      if (pick >= nmax) pick = nmax - 1;
      for (int k = 0; k < cnt; ++k) if (e.edge_N[eb + base + k] == maxn) { if (pick-- == 0) { action = e.edge_action[eb + base + k]; break; } }
    } else {                                                   // no visits at all: uniform over legal moves
      int pick = (int)(u * (double)cnt);
      action = e.edge_action[eb + base + (pick >= cnt ? cnt - 1 : pick)];
    }
  }
  if (action >= 0) apply_action(g, b, w, player, action);    // getNextState with the real player (self_play.py:163)
  player = -player; ++step;
  store_bb<NW>(e.sp_black, gi, e.W, b); store_bb<NW>(e.sp_white, gi, e.W, w);
  e.sp_player[gi] = (int8_t)player; e.sp_step[gi] = step;
  atomicAdd(&e.stats->moves, 1ull);
  int code = ended_code(g, b, w, player);                    // self_play.py:167-168
  if (code != 0) finish_game(e, gi, code);
}

// MCTS.search prologue (mcts.py:288-292) for one game, by its warp: fresh tree, root = node 0 = the pending leaf; the
// search runs `budget` simulations.
template <int NW>
__device__ __forceinline__ void tree_root_game(const EngineDev& e, const Geo<NW>& g, int gi, int lane, int budget) {
  BB<NW> b = load_bb<NW>(e.root_black, gi, e.W) & g.full, w = load_bb<NW>(e.root_white, gi, e.W) & g.full;
  int player = e.root_player[gi] == 1 ? 1 : -1;
  if (lane == 0) {
    e.g_n_nodes[gi] = 1; e.g_n_edges[gi] = 0; e.g_sims_done[gi] = 0; e.g_npending[gi] = 1; e.g_sim_budget[gi] = budget;
    for (int k = 1; k < e.K; ++k) e.leaf_active[gi * e.K + k] = 0;
  }
  publish_leaf<NW>(e, g, gi, lane, gi * e.K, 0, b, w, player, 0);
}

// Rolling self-play: called by the game's warp when the slot has no pending leaf -- either its search has just been
// completed (make the move: sp_move_one) or the slot is waiting for its next root (after a reset, or after a launch
// that ended on its move budget).  Leaves the slot with the root of its next search published as the pending leaf, or
// idle (no budget / no game left in the quota).  Not inlined, arguments by value: the rare path keeps its registers and
// its code out of the persistent kernel's hot loops, and the kernel's parameter structs stay in constant memory.
template <int NW>
__device__ __noinline__ void sp_advance_game(const EngineDev e, const Geo<NW> g, int gi, int lane) {
  int budget = -1;
  if (lane == 0) {
    int left = e.sp_moves_left[gi];
    if (e.sp_phase[gi] && left > 0) {
      sp_move_one<NW>(e, g, gi);
      e.sp_phase[gi] = 0;
      if (left != kMovesUnlimited) e.sp_moves_left[gi] = --left;
    }
    if (!e.sp_phase[gi] && left > 0) {
      budget = sp_prepare_one<NW>(e, g, gi);
      if (budget >= 0) sp_noise_one<NW>(e, g, gi);
    }
  }
  budget = __shfl_sync(kFull, budget, 0);
  if (budget < 0) return;
  __syncwarp();
  tree_root_game<NW>(e, g, gi, lane, budget);
  if (lane == 0) e.sp_phase[gi] = 1;
  __syncwarp();
}

}  // namespace yy
