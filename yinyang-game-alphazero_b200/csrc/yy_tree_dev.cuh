// yy_tree_dev.cuh -- device-side MCTS step of ONE game by ONE warp (shared by the per-step tree kernels in
// yy_tree.cu and the persistent search kernel in yy_fused.cu).
//
// Restates src/yin_yang/ai/mcts.py (Node.expand :50-91, select_child :97-145, update :147-156, _simulate
// :345-414).  Exactness contract: see yy_tree.cu.
#pragma once
#include "yy_engine.cuh"

#include <math.h>

namespace yy {

constexpr unsigned kFull = 0xffffffffu;

template <int NW>
__device__ __forceinline__ int rank_below(const BB<NW>& m, int a) {
  int r = 0;
  int wi = a >> 6, bi = a & 63;
#pragma unroll
  for (int k = 0; k < NW; ++k) {
    if (k < wi) r += popc64(m.w[k]);
    else if (k == wi) r += popc64(m.w[k] & ((1ull << bi) - 1ull));
  }
  return r;
}

// Summary of a child node cached in its parent's edge slot, so that a descent needs ONE dependent memory round trip
// per level (the children's N/W/P and these summaries arrive together):
//   bits [0,32) first edge slot of the child, [32,48) child node id + 1 (0 = not created yet),
//   [48,57) number of children, [57,60) NODE_* flags.
__device__ __forceinline__ uint64_t cmeta_pack(int base, int id, int cnt, int flags) {
  return (uint64_t)(uint32_t)base | ((uint64_t)(uint32_t)(id + 1) << 32) | ((uint64_t)(uint32_t)cnt << 48) | ((uint64_t)(uint32_t)flags << 57);
}
__device__ __forceinline__ int cmeta_base(uint64_t m) { return (int)(uint32_t)m; }
__device__ __forceinline__ int cmeta_child(uint64_t m) { return (int)((m >> 32) & 0xffffu) - 1; }
__device__ __forceinline__ int cmeta_cnt(uint64_t m) { return (int)((m >> 48) & 0x1ffu); }
__device__ __forceinline__ int cmeta_flags(uint64_t m) { return (int)((m >> 57) & 7u); }

__device__ __forceinline__ float terminal_value_f32(int code) {
  // yin_yang_game.py:101-107: +1 / -1 / 0.0001 (Python scalars, weak-promoted to float32 in Node.update)
  return code == 1 ? 1.0f : (code == -1 ? -1.0f : (float)0.0001);
}

// Node.update along a recorded path (mcts.py:406-412): the leaf's own slot gets +v, alternating upwards.
// `vl_pending`: the path already carries a virtual visit and a virtual loss of 1 (multi-leaf mode) -- the visit
// stays, the loss is taken back.
__device__ __forceinline__ void backup_path(const EngineDev& e, const int32_t* path, long long eb, int plen, float v, int lane,
                                            bool vl_pending) {
  for (int i = lane; i < plen; i += 32) {
    long long ei = eb + path[i];
    float sv = ((plen - 1 - i) & 1) ? -v : v;
    if (vl_pending) {
      e.edge_W[ei] = __fadd_rn(__fadd_rn(e.edge_W[ei], 1.0f), sv);
    } else {
      e.edge_N[ei] += 1;
      e.edge_W[ei] = __fadd_rn(e.edge_W[ei], sv);
    }
  }
}

// Writes the state of node `id`, evaluates the rules for it (terminal code + legal mask of the side to
// move) and publishes it in leaf slot `slot` of the evaluation batch.  All lanes hold identical arguments.
template <int NW>
__device__ __forceinline__ void publish_leaf(const EngineDev& e, const Geo<NW>& g, int gi, int lane, int slot, int id,
                                             const BB<NW>& black, const BB<NW>& white, int player, int plen) {
  BB<NW> mask = legal_for(g, black, white, player);
  int code = ended_code_with_mask(g, black, white, player, mask);
  if (lane == 0) {
    long long ni = (long long)gi * e.max_nodes + id;
    store_bb<NW>(e.node_black, ni, e.W, black);
    store_bb<NW>(e.node_white, ni, e.W, white);
    e.node_player[ni] = (int8_t)player;
    e.node_flags[ni] = 0;
    e.node_n_edges[ni] = 0;
    e.node_edge_base[ni] = 0;
    store_bb<NW>(e.leaf_black, slot, e.W, black);
    store_bb<NW>(e.leaf_white, slot, e.W, white);
    store_bb<NW>(e.leaf_mask, slot, e.W, mask);
    e.leaf_code[slot] = (int8_t)code;
    e.leaf_node[slot] = id;
    e.leaf_path_len[slot] = plen;
    e.leaf_active[slot] = 1;
  }
  if (e.evaluator == YY_EVAL_STUB) {  // deterministic-prior mode: evaluator fused into the tree kernel
    uint64_t key = stub_key(g, black, white);
    for (int a = lane; a < e.A; a += 32) e.eval_prior[(long long)slot * e.A + a] = stub_prior(key, a);
    if (lane == 0) e.eval_value[slot] = stub_value(key);
  }
}

// Node.expand (mcts.py:50-91) of the node in `slot` with the evaluator's output + backup of its value.
template <int NW>
__device__ __forceinline__ void expand_and_backup(const EngineDev& e, const Geo<NW>& g, int gi, int lane, int slot, long long nb,
                                                  long long eb, bool multi) {
  const int leaf = e.leaf_node[slot];
  const int code = e.leaf_code[slot];
  const float v = e.eval_value[slot];
  uint8_t flags = NODE_EXPANDED;
  float nodeval = 0.0f;
  int sum_base = 0, sum_cnt = 0;         // what the parent's edge slot will cache about this node
  if (code != 0) {                       // terminal branch (mcts.py:63-68)
    flags |= NODE_TERMINAL; nodeval = terminal_value_f32(code);
  } else {
    BB<NW> mask = load_bb<NW>(e.leaf_mask, slot, e.W);
    int cnt = popcount(mask);
    int base = e.g_n_edges[gi];
    __syncwarp();
    if (cnt > 0 && base + cnt > e.edges_cap) { if (lane == 0) atomicExch(&e.stats->overflow, 1); cnt = 0; }
    if (cnt == 0) {                      // no legal move, not terminal: child-less node, re-evaluated on every
      flags |= NODE_NOCHILD; nodeval = v;  // visit by the reference (is_expanded() stays False) -> same value
    } else {
      const bool noisy = (leaf == 0) && e.noise != nullptr && e.noise_mask != nullptr && e.noise_mask[gi] != 0;
      for (int a = lane; a < e.A; a += 32) {
        if (!test(mask, a)) continue;
        int r = rank_below(mask, a);     // children are created in ascending action order (mcts.py:75-89)
        float p = e.eval_prior[(long long)slot * e.A + a];
        if (noisy) {                     // mcts.py:309-311: f32( f64(f32(f32(1-eps)*p)) + eps*noise_i )
          float keep = __fmul_rn(e.keep_f32, p);
          p = (float)__dadd_rn((double)keep, __dmul_rn(e.eps, e.noise[(long long)gi * e.A + r]));
        }
        long long ei = eb + base + r;
        e.edge_N[ei] = 0; e.edge_W[ei] = 0.0f; e.edge_P[ei] = p; e.edge_cmeta[ei] = 0ull;
        e.edge_action[ei] = (uint8_t)a;
      }
      __syncwarp();
      if (lane == 0) { e.node_edge_base[nb + leaf] = base; e.node_n_edges[nb + leaf] = (int16_t)cnt; e.g_n_edges[gi] = base + cnt; }
      sum_base = base; sum_cnt = cnt;
    }
  }
  const int plen = e.leaf_path_len[slot];
  const int32_t* path = e.leaf_path + (long long)slot * e.max_depth;
  if (lane == 0) {
    e.node_flags[nb + leaf] = flags; e.node_value[nb + leaf] = nodeval; e.leaf_active[slot] = 0;
    if (plen > 0) e.edge_cmeta[eb + path[plen - 1]] = cmeta_pack(sum_base, leaf, sum_cnt, flags);
  }
  // first visit always backs up the evaluator's value (mcts.py:394)
  backup_path(e, path, eb, plen, v, lane, multi && leaf != 0);
  __syncwarp();
}

// One lock-step of every tree: (1) expand the pending leaves with the evaluator's output and back their values
// up (mcts.py:394-412); (2) run simulations from the root until K of them need an evaluation (selection,
// mcts.py:360-362; revisited terminal leaves complete on the spot, :365-367) and publish those leaves.
//   K == 1 : deterministic mode -- exactly the reference's sequential search per game.
//   K  > 1 : throughput mode -- each in-flight simulation leaves a virtual visit and a virtual loss on its path so
//            that the next descent of the same step diverges; a descent that runs into an in-flight node stops.
// `pending_counter` (nullable): incremented by the number of leaves this game published.
// `max_descents` > 0 bounds the simulations started in this call: a game whose simulations keep ending in revisited
// terminals would otherwise hold its warp (and, in the persistent kernel, its whole CTA pair) for many dependent
// descents; it resumes in the next step instead, without a leaf in between (g_npending = -1: "still selecting").
// Returns the number of leaves published; 0 = the search is complete; -1 = still selecting.
template <int NW>
__device__ __forceinline__ int tree_step_game(const EngineDev& e, const Geo<NW>& g, int gi, int lane, int32_t* pending_counter,
                                              int max_descents = 0) {
  const long long nb = (long long)gi * e.max_nodes;
  const long long eb = (long long)gi * e.edges_cap;
  const bool multi = e.K > 1;
  // simulations this search still has to run: its budget (n_sims; fast_sims for a fast self-play search) minus those done
  int left = e.g_sim_budget[gi] - e.g_sims_done[gi];
  int sims_here = 0, evals_here = 0, deepest = 0;

  // ---------------------------------------------------------------- (1) expand + backup
  const int np_in = e.g_npending[gi];
  for (int k = 0; k < np_in; ++k) {
    const int slot = gi * e.K + k;
    const bool is_root = e.leaf_node[slot] == 0;
    expand_and_backup<NW>(e, g, gi, lane, slot, nb, eb, multi);
    if (!is_root) { --left; ++sims_here; }
  }

  // ---------------------------------------------------------------- (2) select
  int np = 0, descents = 0;
  bool blocked = false;
  while (np < left && np < e.K && !blocked) {
    if (max_descents > 0 && descents++ >= max_descents) break;
    const int slot = gi * e.K + np;
    int32_t* path = e.leaf_path + (long long)slot * e.max_depth;
    int node = 0, depth = 0;
    // root summary from the node arrays; every deeper level gets it from the parent's edge slot (cmeta)
    int fl = e.node_flags[nb], base = e.node_edge_base[nb], cnt = e.node_n_edges[nb];
    for (;;) {
      if (!(fl & NODE_EXPANDED)) { blocked = true; break; }  // in-flight node of this step (K > 1 only): give up
      if (fl & (NODE_TERMINAL | NODE_NOCHILD)) {   // revisited terminal (mcts.py:365-367) / child-less node
        __syncwarp();                              // path[] written by lane 0 above
        backup_path(e, path, eb, depth, e.node_value[nb + node], lane, false);
        --left; ++sims_here;
        __syncwarp();
        break;
      }
      // Node.select_child (mcts.py:97-145).  The first 64 children live in registers (two per lane): one round trip.
      const long long e0 = eb + base;
      int n0 = 0, n1 = 0; float w0 = 0.0f, w1 = 0.0f, p0 = 0.0f, p1 = 0.0f; uint64_t m0 = 0ull, m1 = 0ull;
      if (lane < cnt) { n0 = e.edge_N[e0 + lane]; w0 = e.edge_W[e0 + lane]; p0 = e.edge_P[e0 + lane]; m0 = e.edge_cmeta[e0 + lane]; }
      if (lane + 32 < cnt) { n1 = e.edge_N[e0 + lane + 32]; w1 = e.edge_W[e0 + lane + 32]; p1 = e.edge_P[e0 + lane + 32]; m1 = e.edge_cmeta[e0 + lane + 32]; }
      int sum = n0 + n1;
      for (int k = lane + 64; k < cnt; k += 32) sum += e.edge_N[e0 + k];
#pragma unroll
      for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(kFull, sum, off);
      const float sq = (float)sqrt((double)sum);
      float best = -INFINITY; int besti = 0x7fffffff;
      auto consider = [&](int k, int n, float w, float p) {
        const float u = __fdiv_rn(__fmul_rn(__fmul_rn(e.cpuct, p), sq), (float)(1 + n));
        const float q = n > 0 ? __fdiv_rn(w, (float)n) : 0.0f;
        const float ucb = __fadd_rn(q, u);
        if (ucb > best) { best = ucb; besti = k; }
      };
      if (lane < cnt) consider(lane, n0, w0, p0);
      if (lane + 32 < cnt) consider(lane + 32, n1, w1, p1);
      for (int k = lane + 64; k < cnt; k += 32) consider(k, e.edge_N[e0 + k], e.edge_W[e0 + k], e.edge_P[e0 + k]);
#pragma unroll
      for (int off = 16; off; off >>= 1) {
        float ov = __shfl_xor_sync(kFull, best, off); int oi = __shfl_xor_sync(kFull, besti, off);
        if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
      }
      if (besti == 0x7fffffff) besti = 0;
      const int eoff = base + besti;
      uint64_t cm;
      if (besti < 64) {
        const uint64_t mine = (besti & 32) ? m1 : m0;
        cm = __shfl_sync(kFull, mine, besti & 31);
      } else {
        cm = e.edge_cmeta[eb + eoff];
      }
      if (lane == 0) path[depth] = eoff;
      ++depth;
      const int child = cmeta_child(cm);
      if (child < 0) {                      // unexpanded child: getNextState on the parent's state (mcts.py:385-391)
        BB<NW> b = load_bb<NW>(e.node_black, nb + node, e.W), w = load_bb<NW>(e.node_white, nb + node, e.W);
        const int pp = e.node_player[nb + node];
        const int a = e.edge_action[eb + eoff];
        const int id = e.g_n_nodes[gi];
        if (pp == 1) setbit(b, a); else setbit(w, a);   // the slot exists only for a legal action
        __syncwarp();
        if (lane == 0) { e.g_n_nodes[gi] = id + 1; e.edge_cmeta[eb + eoff] = cmeta_pack(0, id, 0, 0); }
        publish_leaf<NW>(e, g, gi, lane, slot, id, b, w, -pp, depth);
        if (multi) {                        // virtual visit + virtual loss along the in-flight path
          __syncwarp();
          for (int i = lane; i < depth; i += 32) {
            long long ei = eb + path[i];
            e.edge_N[ei] += 1;
            e.edge_W[ei] = __fadd_rn(e.edge_W[ei], -1.0f);
          }
        }
        if (depth > deepest) deepest = depth;
        ++np; ++evals_here;
        __syncwarp();
        break;
      }
      node = child; fl = cmeta_flags(cm); base = cmeta_base(cm); cnt = cmeta_cnt(cm);
    }
  }
  __syncwarp();
  const bool selecting = np == 0 && !blocked && left > 0;                 // stopped by max_descents
  if (lane == 0) {
    e.g_sims_done[gi] += sims_here;
    e.g_npending[gi] = selecting ? -1 : np;
    if (np && pending_counter) atomicAdd(pending_counter, np);
    if (sims_here) atomicAdd(&e.stats->sims, (unsigned long long)sims_here);
    if (evals_here) atomicAdd(&e.stats->evals, (unsigned long long)evals_here);
    if (deepest > e.stats->max_depth) atomicMax(&e.stats->max_depth, deepest);
  }
  return selecting ? -1 : np;
}

}  // namespace yy
