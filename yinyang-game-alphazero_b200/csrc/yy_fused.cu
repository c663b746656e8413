// yy_fused.cu -- ONE persistent kernel for a whole MCTS search: residual tower + FC heads + tree step, per CTA.
//
// Games are independent (self_play.py:288-335), so a CTA can own a fixed run of games for the whole search and
// never needs a grid-wide synchronisation: for every simulation it
//   (1) evaluates the pending leaves of its games on the tensor cores -- the residual tower of yy_nn.cu
//       (neural_network.py:94-123) group by group, activations resident in shared memory, then the two FC heads
//       (policy_fc, value_fc1: :112-121) for all of its <= 32 boards at once, the FC weights streamed through the
//       same bulk-copy ring as the conv weights and used as the M = 128 UMMA operand (boards are the N operand);
//   (2) finishes the heads on the CUDA cores (softmax over all A logits, predict() :152; value_fc2 + tanh :121);
//   (3) runs Node.expand / backup / select (mcts.py:50-156, 345-414) for each of its games, one warp per game
//       (tree_step_game, yy_tree_dev.cuh), which publishes the next leaves.
// Nothing returns to the host between simulations: a search is one launch instead of 4 x (n_sims + 1).
// The same kernel with iterations = 1 and the tree step off is the batched network forward (yy_evaluate).
//
// Within a layer the tiles of a group run SKEWED (see `skewed` below): the issuer walks the last and the first two weight stages
// of a layer tile by tile, so a tile's epilogue runs under the other tiles' MMAs instead of next to their epilogues.
// Warp roles: warp 0 weight producer, warp 1 MMA issuer, warps 2-17 epilogue / heads / tree, warps 18-19 background
// selection (simulations that end in revisited terminals need no evaluation, mcts.py:365-367: games in such a stretch
// are advanced here, concurrently with the tower, instead of holding up the tree phase of their CTA pair).
// Roofline: tensor (the tower's conv MMAs are > 99 % of the FLOPs; see yy_nn.cu for the tower layout).
#include "yy_nn.cuh"
#include "yy_tower.cuh"
#include "yy_selfplay_dev.cuh"

namespace yy {
using namespace ptx;

struct FusedArgs {
  TowerGeo g;
  FcGeo fc;
  const uint8_t* conv_stream;  // stage-ordered bf16 conv weight blocks (CTA-pair kernel: each stage split in two N halves)
  const float* conv_bias;      // [1 + 2*blocks][128] then head [64]
  const uint8_t* fc_stream;    // stage-ordered bf16 FC weight blocks (policy_fc, value_fc1)
  const float* fc_policy_b; const float* fc_value1_b; const float* fc_value2_w; const float* fc_value2_b;
  const uint64_t* black; const uint64_t* white;   // [count][W] boards to evaluate (search: the leaf batch)
  long long count;
  int boards_per_cta;          // contiguous run of boards (= games in a search) owned by a CTA
  // arena: the grid is two halves of whole CTA pairs; CTAs [half_grid, grid) own boards [half_count, count) and stream the
  // weight image at byte offset wb_off from the one above (same layout).  Other modes: half_grid = grid, half_count = count.
  int half_grid;
  long long half_count;
  long long wb_off;
  int batch_boards;            // <= FC_N boards per heads pass (whole groups of g.Gb boards, except possibly the last group)
  __nv_bfloat16* headfeat;     // [count][64*A] head-conv features, index c*A + cell (L2-resident round trip)
  float* policy; float* value; float* logits;     // [count][A], [count], optional [count][A]
  int iterations;              // 1 = plain forward; n_sims + 1 = whole search; rolling self-play: any number of steps
  int mode;                    // YY_FUSED_FORWARD / YY_FUSED_SEARCH (tree step after every evaluation) / YY_FUSED_SELFPLAY / YY_FUSED_ARENA
  int use_nn;                  // 0 = deterministic-prior (stub) evaluator: tree steps only
  int no_skew;                 // developer A/B (yy_engine_set_debug_flags bit 1): tiles of a group in lock step as in round 1
  int split_halves;            // developer A/B (yy_engine_set_debug_flags bit 0): the two halves of a group ping-pong through the
                               // tensor cores.  OFF in the product: it hides the epilogue (the MMA issuer's wait for activations
                               // drops from 513 k to 93 k cycles per step) but every half streams the layer's weights again, and
                               // the weight stream (~10 B/clk per SM through the 3-slot ring) then stalls the issuer for 735 k
                               // cycles per step: 1,286 against 1,298 TFLOP/s (profiles/r02_ab_pingpong_*.txt)
  // symmetric evaluation (FormSpec, yy_nn.cuh): the form a board is evaluated in.  Averaging walks n_avg entries per
  // board, one per form (entry i -> board i / n_avg, form i % n_avg); the heads pass averages them in ascending form order.
  int form_mode, form_fixed, n_avg;
  uint64_t form_seed;
  long long* dbg;
};

__device__ __forceinline__ void st_cluster_u32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}

constexpr int kEpiBarrier = 1;   // named barrier of the 16 epilogue warps
constexpr int kTreeBarrier = 2;  // epilogue + background selection warps: every tree step of the CTA is done
__device__ __forceinline__ void epi_sync() { asm volatile("bar.sync %0, %1;" ::"n"(kEpiBarrier), "n"(TW_EPI_THREADS) : "memory"); }
__device__ __forceinline__ void tree_sync() { asm volatile("bar.sync %0, %1;" ::"n"(kTreeBarrier), "n"(TW_EPI_THREADS + 32 * TW_BG_WARPS) : "memory"); }

// CG = 1: one CTA per SM, M = 128 MMAs.  CG = 2: CTA pairs (cluster of 2, tcgen05 cta_group::2): the leader issues M = 256
// MMAs over both CTAs' activation tiles, each CTA stages only its half of the weight slice's output channels -- halves
// the weight bytes every SM pulls from L2 and takes the B-operand fetch off the shared-memory port, which a 128x128x16
// SS-MMA otherwise saturates (8 KB per 64 cycles = 128 B/clk).
template <int NW, int CG>
__global__ void __launch_bounds__(TW_THREADS, 1) fused_kernel(const FusedArgs a, const EngineDev e, const Geo<NW> geo) {
  extern __shared__ __align__(128) uint8_t smem[];
  const TowerGeo& g = a.g;
  const FcGeo& fc = a.fc;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int L = 2 * g.blocks + 2;  // stem + 2*blocks tower convs + head conv
  int16_t* pos_p = reinterpret_cast<int16_t*>(smem + SM_POS);                       // M row -> padded position
  int16_t* pos_tab = reinterpret_cast<int16_t*>(smem + SM_POS + 128 * TW_MAXT * 2);    // M row -> board*256 + cell, or -1
  const uint32_t bar0 = smem_u32(smem + SM_BAR);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (TW_NBAR + s); };
  auto peer_full_bar = [&](int s) { return bar0 + 8u * (2 * TW_NBAR + s); };   // leader: the follower's stage s landed
  // accumulators complete / activations ready, one pair per HALF of a group (developer A/B split_halves: the two halves of
  // a group ping-pong through the tensor cores; the product runs a group as ONE half)
  auto acc_full = [&](int h) { return bar0 + 8u * (3 * TW_NBAR + 2 * h); };
  auto act_ready = [&](int h) { return bar0 + 8u * (3 * TW_NBAR + 2 * h + 1); };
  // the same pair per TILE for groups whose tiles are skewed against each other (see `skewed` below)
  auto acc_full_t = [&](int t) { return bar0 + 8u * (3 * TW_NBAR + 4 + 2 * t); };
  auto act_ready_t = [&](int t) { return bar0 + 8u * (3 * TW_NBAR + 4 + 2 * t + 1); };
  const int rank = CG == 2 ? (int)cluster_ctarank() : 0;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM_TMEM);

  // ---- one-time setup ----
  for (int i = tid; i < (SM_POS - SM_ACT) / 4; i += TW_THREADS) reinterpret_cast<uint32_t*>(smem + SM_ACT)[i] = 0u;   // act + ring
  for (int i = tid; i < 128 * TW_MAXT; i += TW_THREADS) {
    int p, v;
    tower_row(g, i, p, v);
    pos_p[i] = (int16_t)p;
    pos_tab[i] = (int16_t)v;
  }
  if (tid == 0) {
    for (int s = 0; s < TW_NBAR; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); mbar_init(peer_full_bar(s), 1); }
    for (int h = 0; h < 2; ++h) {
      mbar_init(acc_full(h), 1);
      mbar_init(act_ready(h), CG * TW_EPI_THREADS);   // pair: the leader's barrier also collects the follower's epilogue threads
    }
    for (int t = 0; t < TW_MAXT; ++t) { mbar_init(acc_full_t(t), 1); mbar_init(act_ready_t(t), CG * 128); }   // a tile has 4 epilogue warps per CTA
    fence_barrier_init();
  }
  if (warp == 1) { if (CG == 2) tmem_alloc2(smem_u32(tmem_slot), 512); else tmem_alloc(smem_u32(tmem_slot), 512); }
  fence_proxy_async_smem();
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (a.dbg && tid == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); a.dbg[128 + 2 * blockIdx.x] = (long long)gt; }
  const uint32_t act_base = smem_u32(smem + SM_ACT);
  const uint32_t ring_base = smem_u32(smem + SM_RING);
  // This CTA owns the run of boards [run_lo, run_lo + my_len).  A plain forward walks the whole run; a search / self-play
  // step walks only the games that have a pending leaf, compacted into e.act_list by the epilogue warps at the end of the
  // previous step (a game whose remaining simulations ended in revisited terminals has none: mcts.py:365-367 makes no
  // predict call there, so no tensor time is spent on it).  The walk goes in batches of <= FC_N boards, a batch in groups
  // of Gb boards.  In a pair both CTAs must walk the same batches / groups / tiles: the structure comes from the larger of
  // the two counts; entries past a CTA's own count are padding.
  auto clampl = [](long long v, long long hi) { return v < 0 ? 0 : (v > hi ? hi : v); };
  // (arena: both CTAs of a pair are in the same half, so they stream the same image and share the structural length)
  const int half = (int)blockIdx.x >= a.half_grid ? 1 : 0, cta = (int)blockIdx.x - half * a.half_grid;
  const long long run_lo = half * a.half_count + (long long)cta * a.boards_per_cta;
  const int my_len = (int)clampl(a.half_count - (long long)cta * a.boards_per_cta, a.boards_per_cta);
  const int st_len = (int)clampl(a.half_count - (long long)(cta - rank) * a.boards_per_cta, a.boards_per_cta);
  const long long wofs = half ? a.wb_off : 0;    // weight image of this CTA pair: byte offset from image A
  auto wf = [&](const float* p) { return reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(p) + wofs); };
  const bool dyn = a.mode != YY_FUSED_FORWARD;
  volatile int* cnt_s = reinterpret_cast<volatile int*>(smem + SM_CNT);   // [step parity][cluster rank][leaves, selecting]
  const int E = a.n_avg;                         // walk entries per board (1 unless forms are averaged)
  int n_mine = my_len * E, n_struct = st_len * E;   // my real entries / structural length of this step's walk
  int n_sel = 0;                                 // my games whose search continues without a leaf in this step
  bool any_work = true;
  // every thread of the CTA (pair): wait for the counts of step `iter` (written by the compaction of the step before)
  auto fetch_counts = [&](int iter) {
    if (CG == 2) cluster_sync_all(); else asm volatile("bar.sync 0;" ::: "memory");
    volatile int* c = cnt_s + (iter & 1) * 4;
    const int c0 = c[0] * E, c1 = CG == 2 ? c[2] * E : 0, s0 = c[1], s1 = CG == 2 ? c[3] : 0;
    n_mine = rank ? c1 : c0; n_struct = c0 > c1 ? c0 : c1; n_sel = rank ? s1 : s0;
    any_work = (c0 | c1 | s0 | s1) != 0;
  };
  // tiles a group starting at entry b0 needs when its batch ends at `lim`
  // (+pitch+1: the taps of the last real position read that far; rows beyond the group's tiles may be stale)
  auto tiles_for = [&](int b0, int lim) {
    int nb = lim - b0; if (nb > g.Gb) nb = g.Gb;
    return tower_tiles_for(g, nb);
  };
  // A group's tiles split into two halves that are INDEPENDENT through the whole tower (no 3x3 tap of one half reads a
  // row of the other): interleaved pairs (8x8: a tile = two whole boards, zero row groups between tiles) and half-board
  // tiles (16x16: two tiles = one board).  Returns the tiles of half 0; == T: one half only (other layouts, tiny groups).
  auto half_split = [&](int T) {
    if (!a.split_halves) return T;
    if (g.row_aligned == 3) return T >= 2 ? (T + 1) >> 1 : T;
    if (g.row_aligned == 2) return T == 4 ? 2 : T;
    return T;
  };
  // Tile skew.  In a layer every weight stage serves all tiles of the group, so the tiles used to finish the layer together: their
  // epilogues then ran side by side while the tensor cores idled (26 % of a step), and the next layer started for all of them at
  // once.  When the tiles of a group are independent through the tower (interleaved layouts: no tap of a tile reads a row of
  // another; half-board tiles: in units of the two halves of a board), the MMA issuer instead walks the LAST and the FIRST TW_SKEW stages of a layer tile by tile (they fit the ring
  // together) and only the stages in between stage by stage: tile 0 completes the layer TW_SKEW * (T - 1) stage-tiles of MMA time
  // before tile T-1, its epilogue runs under the other tiles' MMAs, and it starts the next layer as soon as ITS activations are
  // in place.  Weights are still streamed once per layer and group.  Synchronisation is per tile (acc_full_t / act_ready_t).
  static_assert(TW_SKEW <= TW_STAGES, "the tile-by-tile stages of a layer must fit the weight ring together");
  auto skewed = [&](int T) { return !a.split_halves && !a.no_skew && (g.row_aligned == 2 ? T == 4 : (g.row_aligned == 3 || g.row_aligned == 4) && T >= 3); };
  auto batch_end = [&](int bb0) { return (bb0 + a.batch_boards < n_struct) ? bb0 + a.batch_boards : n_struct; };   // structural
  // FC stage geometry: rows of M tile t of head h
  auto fc_tiles = [&](int h) { return h ? 2 : fc.Tp; };
  auto fc_rows = [&](int h, int t) { return (h || t < fc.Tp - 1) ? 128 : fc.Rp_last; };
  auto panel_stages = [&](int p) { const int r = fc.KS - p * FC_PANEL_STAGES; return r < FC_PANEL_STAGES ? r : FC_PANEL_STAGES; };
  // Weight slots: the conv stream cycles through the TW_STAGES ring slots; the FC stream of a batch cycles through
  // TW_FC_SLOTS slots -- the ring plus two more in the tail of the activation region, which is free while the heads run
  // (the FC phase is bound by the bytes in flight: 16 KB per slot against ~1 us of L2 latency).  Every role tracks one
  // phase bit per slot, so the two cycles can share the ring.  A policy tile of <= 64 rows packs two K = 64 stages per slot.
  auto slot_addr = [&](uint32_t s) {
    return s < (uint32_t)TW_STAGES ? ring_base + s * TW_STAGE_BYTES : act_base + (uint32_t)TW_FC_EXTRA_OFF + (s - TW_STAGES) * TW_STAGE_BYTES;
  };
  auto fc_merge = [&](int h, int t) { return fc_rows(h, t) <= 64 ? 2 : 1; };
  // the tower's view of the ring: TW_CONV_SLOTS slots of 8 KB; barrier set s serves conv slot s and FC slot s (the two
  // cycles never overlap in time: the producer waits for the last MMA of one before it starts the other)
  auto conv_slot_addr = [&](uint32_t s) { return ring_base + s * (uint32_t)TW_CONV_SLOT_BYTES; };

  if (warp == 0) {
    // =========================================================== weight producer (whole warp walks the loop with
    // warp-uniform state; one elected lane issues the bulk copies -- keeps everything on the uniform datapath)
    if (!a.use_nn) {
      for (int iter = 0; dyn && iter < a.iterations; ++iter) { fetch_counts(iter); if (!any_work) break; }
    } else {
      uint32_t ci = 0, used = 0, ephase = 0, acc_n[2] = {0, 0};     // conv stage counter, slots used so far, empty-phase bits, commits so far per half
      uint32_t acc_nt[TW_MAXT] = {0, 0, 0, 0};                      // commits so far per tile (skewed groups)
      int last_skew_T = 0;                                          // > 0: the batch's last group was skewed and had this many tiles
      auto push_to = [&](uint32_t slot, uint32_t dst, const uint8_t* src, uint32_t bytes) {
        if ((used >> slot) & 1u) { mbar_wait(empty_bar(slot), (ephase >> slot) & 1u); ephase ^= 1u << slot; }
        used |= 1u << slot;
        if (elect_one()) {
          mbar_arrive_expect_tx(full_bar(slot), bytes);
          bulk_g2s(dst, src, bytes, full_bar(slot));
        }
        __syncwarp();
      };
      auto push = [&](uint32_t slot, const uint8_t* src, uint32_t bytes) { push_to(slot, slot_addr(slot), src, bytes); };
      bool fc_before = false;
      // pair, FC stages: both CTAs need the SAME weight tile, so the two producers take turns fetching a stage and the
      // copy is multicast into both CTAs' slots (each CTA arms its own barrier) -- halves the L2 reads of the FC phase,
      // which is bound by the aggregate L2 bandwidth (all SMs stream the 1.25 MB at the same time).  A slot is free in
      // both CTAs at once: its empty barrier is armed by the leader's multicast commit.
      auto push_shared = [&](uint32_t slot, const uint8_t* src, uint32_t bytes, bool mine) {
        if ((used >> slot) & 1u) { mbar_wait(empty_bar(slot), (ephase >> slot) & 1u); ephase ^= 1u << slot; }
        used |= 1u << slot;
        if (elect_one()) {
          mbar_arrive_expect_tx(full_bar(slot), bytes);
          if (mine) bulk_g2s_multicast(slot_addr(slot), src, bytes, full_bar(slot), (uint16_t)3);
        }
        __syncwarp();
      };
      for (int iter = 0; iter < a.iterations; ++iter) {
        if (dyn) { fetch_counts(iter); if (!any_work) break; }
        for (int bb0 = 0; bb0 < n_struct; bb0 += a.batch_boards) {
          const int slim = batch_end(bb0);
          int nh = 1;
          // the FC heads of the previous batch used the ring as 16 KB slots: their last MMA must be complete before 8 KB
          // conv slots (a different carving of the same memory) are filled again
          if (TW_CONV_SLOT_BYTES != TW_STAGE_BYTES && fc_before) mbar_wait(acc_full(0), (acc_n[0] - 1) & 1u);
          for (int b0 = bb0; b0 < slim; b0 += g.Gb) {
            const int T = tiles_for(b0, slim);
            nh = half_split(T) < T ? 2 : 1;
            const bool skew = skewed(T);
            last_skew_T = skew ? T : 0;
            for (int l = 0; l < L; ++l) {
              const LayerInfo li = layer_info(l, g.blocks, CG);
              const uint32_t bytes = (uint32_t)li.stage_bytes / CG;     // pair: my half of the stage's output channels
              const uint8_t* src = a.conv_stream + wofs + li.stream_off + (long long)rank * bytes;
              if (skew) {
#pragma unroll
                for (int t = 0; t < TW_MAXT; ++t) if (t < T) ++acc_nt[t];
              }
              for (int hh = 0; hh < nh; ++hh) {                          // every half of the group streams the layer's weights
                if (!skew) ++acc_n[hh];
                for (int j = 0; j < li.n_stages; ++j, ++ci)
                  push_to(ci % TW_CONV_SLOTS, conv_slot_addr(ci % TW_CONV_SLOTS), src + (long long)j * li.stage_bytes, bytes);
              }
            }
          }
          // the extra FC slots overlay activation rows: wait until the last head conv of the batch has been computed, in
          // both halves (commit number acc_n - 1 of acc_full; it cannot be overtaken -- the next commit needs stages from me)
          if (last_skew_T) {                                           // skewed group: its last tile's last commit covers every MMA before it
            uint32_t n_last = 0;
#pragma unroll
            for (int t = 0; t < TW_MAXT; ++t) if (t == last_skew_T - 1) n_last = acc_nt[t];
            mbar_wait(acc_full_t(last_skew_T - 1), (n_last - 1) & 1u);
          } else {
            mbar_wait(acc_full(0), (acc_n[0] - 1) & 1u);
            if (nh == 2) mbar_wait(acc_full(1), (acc_n[1] - 1) & 1u);
          }
          const uint8_t* src = a.fc_stream + wofs;
          uint32_t fi = 0;
          fc_before = true;
          for (int h = 0; h < 2; ++h)
            for (int p = 0; p < fc.n_panels; ++p, ++acc_n[0]) {
              const int ns = panel_stages(p);
              for (int t = 0; t < fc_tiles(h); ++t) {
                const uint32_t bytes = 128u * (uint32_t)fc_rows(h, t);
                const int mg = fc_merge(h, t);
                for (int s0 = 0; s0 < ns; s0 += mg, ++fi) {
                  const uint32_t k = (uint32_t)(ns - s0 < mg ? ns - s0 : mg);
                  if (CG == 2) push_shared(fi % TW_FC_SLOTS, src, k * bytes, (fi & 1u) == (uint32_t)rank);
                  else push(fi % TW_FC_SLOTS, src, k * bytes);
                  src += k * bytes;
                }
              }
            }
        }
      }
    }
  } else if (warp == 1) {
    // =========================================================== MMA issuer (whole warp runs the control flow, the
    // tcgen05.mma / commit instructions are issued by one elected lane; descriptors are base + constant deltas)
    if (!a.use_nn) {
      for (int iter = 0; dyn && iter < a.iterations; ++iter) { fetch_counts(iter); if (!any_work) break; }
    } else if (rank != 0) {
      // follower of a pair: no MMAs to issue -- relay "my half of stage s has landed" to the leader's peer-full ring
      uint32_t ci = 0, fphase = 0;
      auto relay = [&](uint32_t slot) {
        mbar_wait(full_bar(slot), (fphase >> slot) & 1u); fphase ^= 1u << slot;
        if (elect_one()) mbar_arrive_cluster(mapa_u32(peer_full_bar(slot), 0));
        __syncwarp();
      };
      for (int iter = 0; iter < a.iterations; ++iter) {
        if (dyn) { fetch_counts(iter); if (!any_work) break; }
        for (int bb0 = 0; bb0 < n_struct; bb0 += a.batch_boards) {
          const int slim = batch_end(bb0);
          for (int b0 = bb0; b0 < slim; b0 += g.Gb) {
            const int T = tiles_for(b0, slim);
            const int nh = half_split(T) < T ? 2 : 1;
            for (int l = 0; l < L; ++l) { const int ns = nh * layer_info(l, g.blocks, CG).n_stages; for (int j = 0; j < ns; ++j, ++ci) relay(ci % TW_CONV_SLOTS); }
          }
          uint32_t fi = 0;
          for (int h = 0; h < 2; ++h)
            for (int p = 0; p < fc.n_panels; ++p)
              for (int t = 0; t < fc_tiles(h); ++t) {
                const int ns = (panel_stages(p) + fc_merge(h, t) - 1) / fc_merge(h, t);
                for (int j = 0; j < ns; ++j, ++fi) relay(fi % TW_FC_SLOTS);
              }
        }
      }
    } else {
      uint32_t ci = 0, fphase = 0, act_phase[2] = {0, 0}, actt_phase = 0;   // actt_phase bit t: parity of act_ready_t(t)
      long long stall_w = 0, stall_a = 0, t_start = clock64();     // developer stamps: cycles the issuer waited for weights / activations
      auto wait_stage = [&](uint32_t slot) {
        const uint32_t parity = (fphase >> slot) & 1u;
        fphase ^= 1u << slot;
        const long long t0 = a.dbg ? clock64() : 0;
        mbar_wait(full_bar(slot), parity);
        if (CG == 2) mbar_wait_cluster(peer_full_bar(slot), parity);
        if (a.dbg) stall_w += clock64() - t0;
      };
      auto wait_act = [&](int h) {
        const long long t0 = a.dbg ? clock64() : 0;
        if (CG == 2) mbar_wait_cluster(act_ready(h), act_phase[h]); else mbar_wait(act_ready(h), act_phase[h]);
        act_phase[h] ^= 1;
        if (a.dbg) stall_a += clock64() - t0;
      };
      auto wait_act_t = [&](int t) {
        const long long t0 = a.dbg ? clock64() : 0;
        const uint32_t parity = (actt_phase >> t) & 1u;
        if (CG == 2) mbar_wait_cluster(act_ready_t(t), parity); else mbar_wait(act_ready_t(t), parity);
        actt_phase ^= 1u << t;
        if (a.dbg) stall_a += clock64() - t0;
      };
      auto mma = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
        if (CG == 2) tc_mma_bf16_2(d, ad, bd, idesc, acc); else tc_mma_bf16(d, ad, bd, idesc, acc);
      };
      auto commit = [&](uint32_t bar) { if (CG == 2) tc_commit2(bar); else tc_commit(bar); };
      uint64_t tile_delta[TW_MAXT];                                // start of M=128 tile t, in 16-byte rows
#pragma unroll
      for (int t = 0; t < TW_MAXT; ++t)
        tile_delta[t] = (uint64_t)tower_tile_start(g, t);
      constexpr uint64_t kK16DeltaA = (2u * TW_ROWS * 16u) >> 4;   // next K=16 slice: +2 channel chunks
      constexpr uint64_t kK16DeltaF = (2u * FC_LBO) >> 4;          // same for the FC feature panel
      for (int iter = 0; iter < a.iterations; ++iter) {
        if (dyn) { fetch_counts(iter); if (!any_work) break; }
        for (int bb0 = 0; bb0 < n_struct; bb0 += a.batch_boards) {
          const int slim = batch_end(bb0);
          for (int b0 = bb0; b0 < slim; b0 += g.Gb) {
            const int T = tiles_for(b0, slim);
            const int T0 = half_split(T), nh = T0 < T ? 2 : 1;
            const bool skew = skewed(T);
            for (int l = 0; l < L; ++l) {
              const LayerInfo li = layer_info(l, g.blocks, CG);
              const bool preloaded = (l >= 1 && l <= 2 * g.blocks && (l & 1) == 0);  // conv2: accumulator holds the skip input
              const uint32_t idesc = idesc_bf16(128 * CG, li.N);
              const uint32_t nrows_b = (uint32_t)li.N / CG;                          // weight rows staged per CTA
              const uint64_t k16_delta_b = (uint64_t)((2u * nrows_b * 16u) >> 4);
              if (skew) {
                // stages [0, head) and [NS - tail, NS) tile by tile, the ones in between stage by stage; a short layer (the head
                // convolution: one stage) is all tail
                const int NS = li.n_stages;
                const int head = NS >= 2 * TW_SKEW ? TW_SKEW : 0, tail = NS >= 2 * TW_SKEW ? TW_SKEW : NS;
                const uint32_t ci0 = ci;
                uint32_t waited = 0;                                                 // bit j: stage j of this layer has landed (both CTAs)
                auto stage_ready = [&](int j) {
                  if (!((waited >> j) & 1u)) { wait_stage((ci0 + (uint32_t)j) % TW_CONV_SLOTS); tc_fence_after(); waited |= 1u << j; }
                };
                auto issue = [&](int t, int j) {
                  const uint32_t slot = (ci0 + (uint32_t)j) % TW_CONV_SLOTS;
                  int tapshift, chunk0;
                  stage_info(l, j, g.blocks, g.pitch, g.dy_rows, CG, tapshift, chunk0);
                  const uint64_t ad0 = smem_desc(act_base + (uint32_t)((chunk0 * TW_ROWS + TW_PAD + tapshift) * 16), TW_ROWS * 16, (uint32_t)g.sbo_bytes) +
                                       (uint64_t)tower_tile_start(g, t);
                  const uint64_t bd0 = smem_desc(conv_slot_addr(slot), nrows_b * 16, 128);
                  const uint32_t acc0 = (preloaded || j > 0) ? 1u : 0u;
                  if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < 4 * CG; ++k)
                      if (k < li.nk16)
                        mma(tmem_base + (uint32_t)(t * 128), ad0 + (uint64_t)k * kK16DeltaA, bd0 + (uint64_t)k * k16_delta_b, idesc, k > 0 ? 1u : acc0);
                  }
                  __syncwarp();
                };
                auto free_stage = [&](int j) { if (elect_one()) commit(empty_bar((ci0 + (uint32_t)j) % TW_CONV_SLOTS)); __syncwarp(); };
                // U tiles form a unit that must move together: 1 when tiles are independent, 2 for half-board tiles (a tap of one half
                // reads the other half's boundary column, and the epilogue overwrites activations in place)
                const int U = g.row_aligned == 2 ? 2 : 1;
                for (int u0 = 0; u0 < T && head > 0; u0 += U) {
                  for (int t = u0; t < u0 + U && t < T; ++t) wait_act_t(t);
                  tc_fence_after();
                  for (int t = u0; t < u0 + U && t < T; ++t)
                    for (int j = 0; j < head; ++j) { stage_ready(j); issue(t, j); if (t == T - 1) free_stage(j); }
                }
                for (int j = head; j < NS - tail; ++j) {
                  stage_ready(j);
                  for (int t = 0; t < T; ++t) issue(t, j);
                  free_stage(j);
                }
                for (int u0 = 0; u0 < T; u0 += U) {
                  if (head == 0) {                                                   // the unit's first MMAs of this layer
                    for (int t = u0; t < u0 + U && t < T; ++t) wait_act_t(t);
                    tc_fence_after();
                  }
                  for (int t = u0; t < u0 + U && t < T; ++t)
                    for (int j = NS - tail; j < NS; ++j) { stage_ready(j); issue(t, j); if (t == T - 1) free_stage(j); }
                  for (int t = u0; t < u0 + U && t < T; ++t) { if (elect_one()) commit(acc_full_t(t)); __syncwarp(); }
                }
                ci += (uint32_t)NS;
                continue;
              }
             for (int hh = 0; hh < nh; ++hh) {
              const int tlo = hh ? T0 : 0, thi = hh ? T : T0;
              wait_act(hh);
              tc_fence_after();
              for (int j = 0; j < li.n_stages; ++j, ++ci) {
                const uint32_t slot = ci % TW_CONV_SLOTS;
                int tapshift, chunk0;
                stage_info(l, j, g.blocks, g.pitch, g.dy_rows, CG, tapshift, chunk0);
                wait_stage(slot);
                tc_fence_after();
                const uint64_t ad0 = smem_desc(act_base + (uint32_t)((chunk0 * TW_ROWS + TW_PAD + tapshift) * 16), TW_ROWS * 16, (uint32_t)g.sbo_bytes);
                const uint64_t bd0 = smem_desc(conv_slot_addr(slot), nrows_b * 16, 128);
                const uint32_t acc0 = (preloaded || j > 0) ? 1u : 0u;
                if (elect_one()) {
#pragma unroll
                  for (int t = 0; t < TW_MAXT; ++t) {
                    if (t >= tlo && t < thi) {
#pragma unroll
                      for (int k = 0; k < 4 * CG; ++k) {
                        if (k < li.nk16)
                          mma(tmem_base + (uint32_t)(t * 128), ad0 + tile_delta[t] + (uint64_t)k * kK16DeltaA,
                              bd0 + (uint64_t)k * k16_delta_b, idesc, k > 0 ? 1u : acc0);
                      }
                    }
                  }
                  commit(empty_bar(slot));
                }
                __syncwarp();
              }
              if (elect_one()) commit(acc_full(hh));
              __syncwarp();
             }
            }
          }
          // ---- FC heads: D[o][board] (+)= Wfc[o][k] * feat[board][k]; A = weight stage in the ring, B = feature panel
          // (pair: both CTAs stage the same weight tile, so both get D for all 2 x FC_N boards; column block `rank` is mine)
          const uint32_t idesc_fc = idesc_bf16(128 * CG, FC_N * CG);
          uint32_t fi = 0;
          for (int h = 0; h < 2; ++h)
            for (int p = 0; p < fc.n_panels; ++p) {
              const int ns = panel_stages(p);
              wait_act(0);
              tc_fence_after();
              for (int t = 0; t < fc_tiles(h); ++t) {
                const uint32_t R = (uint32_t)fc_rows(h, t);
                const uint32_t dcol = (uint32_t)((h ? fc.Tp + t : t) * FC_N * CG);
                const uint64_t k16_delta_w = (uint64_t)((2u * R * 16u) >> 4);
                const int mg = fc_merge(h, t);
                for (int s0 = 0; s0 < ns; s0 += mg, ++fi) {
                  const uint32_t slot = fi % TW_FC_SLOTS;
                  const int nk = 4 * (ns - s0 < mg ? ns - s0 : mg);      // K = 16 slices in this slot
                  wait_stage(slot);
                  tc_fence_after();
                  const uint64_t wd0 = smem_desc(slot_addr(slot), R * 16, 128);
                  const uint64_t fd0 = smem_desc(act_base + (uint32_t)(s0 * 8 * FC_LBO), FC_LBO, 128);
                  const uint32_t acc0 = (p > 0 || s0 > 0) ? 1u : 0u;
                  if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                      if (k < nk)
                        mma(tmem_base + dcol, wd0 + (uint64_t)k * k16_delta_w, fd0 + (uint64_t)k * kK16DeltaF, idesc_fc, k > 0 ? 1u : acc0);
                    commit(empty_bar(slot));
                  }
                  __syncwarp();
                }
              }
              if (elect_one()) commit(acc_full(0));
              __syncwarp();
            }
        }
      }
      if (a.dbg && lane == 0 && blockIdx.x == 0) { a.dbg[920] = stall_w; a.dbg[921] = stall_a; a.dbg[922] = clock64() - t_start; }
    }
  } else if (warp >= 2 + TW_EPI_WARPS) {
    // =========================================================== background selection warps: while the tower runs, they
    // advance the games of my run that are "still selecting" (tree_step_game stopped on max_descents without reaching a
    // leaf that needs an evaluation), one simulation at a time, until the game has a leaf (or has completed its search:
    // then its move and the root of its next search) or the epilogue warps reach this step's tree phase.
    const int bw = warp - 2 - TW_EPI_WARPS;
    volatile int* stop = cnt_s + 8;
    for (int iter = 0; dyn && iter < a.iterations; ++iter) {
      fetch_counts(iter);
      if (!any_work) break;
      if (n_struct > 0) {       // (without a tower pass the epilogue warps take these games themselves)
        const int32_t* sel = e.act_list + run_lo + my_len - 1;
        for (int k = bw; k < n_sel; k += TW_BG_WARPS) {
          const int gi = sel[-k];
          do {      // at least one simulation per game and step: a search of S simulations ends within 2 (S + 1) steps
            const int np = tree_step_game<NW>(e, geo, gi, lane, nullptr, 1);
            if (np == 0 && a.mode >= YY_FUSED_SELFPLAY) advance_game<NW>(e, geo, gi, lane, a.mode);
            if (np != -1) break;
          } while (*stop != iter + 1);
        }
      }
      if (iter + 1 < a.iterations) tree_sync();
    }
  } else {
    // =========================================================== epilogue warps (2..17): warp -> (tile, lane quarter)
    const int ew = warp - 2;
    const int etid = tid - 64;
    const int quarter = warp & 3;        // TMEM lanes a warp may touch: 32*(warp_id % 4) ..
    const int tile0 = ew >> 2;           // with 16 warps every tile of the group has its own 4 warps
    constexpr int kTileStride = TW_EPI_WARPS / 4;
    uint32_t acc_phase[2] = {0, 0}, acct_phase = 0;     // acct_phase bit t: parity of acc_full_t(t) (skewed groups)
    uint8_t* act = smem + SM_ACT;
    float* sc_logit = reinterpret_cast<float*>(act);                 // [FC_N][256] heads scratch (act region is free then)
    float* sc_hidden = reinterpret_cast<float*>(act) + FC_N * 256;   // [FC_N][256] relu(fc1) * w2
    float* bias_s = reinterpret_cast<float*>(smem + SM_BIAS);
    // developer stamps: tower / FC / heads+tree / barrier / zero, and inside FC: feature-panel loads / MMA waits / scatter
    long long ph_t = clock64(), ph_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sub_t = 0;
    auto phase = [&](int k) { if (a.dbg) { const long long now = clock64(); ph_acc[k] += now - ph_t; ph_t = now; sub_t = now; } };
    auto sub = [&](int k) { if (a.dbg) { const long long now = clock64(); ph_acc[k] += now - sub_t; sub_t = now; } };
    const uint32_t act_ready_leader[2] = {CG == 2 ? mapa_u32(act_ready(0), 0) : act_ready(0), CG == 2 ? mapa_u32(act_ready(1), 0) : act_ready(1)};
    const int sub4 = ew >> 2;            // which of the 4 warps that share my TMEM lane quarter
    // Accumulators complete: ONE warp polls the mbarrier, the other 15 block on the hardware named barrier.  (With all
    // 16 warps spinning on try_wait for the 80 % of a layer that the MMAs take, the poll loop was 70 % of all executed
    // instructions of the kernel; measured effect on the step time: within noise, -0.5 % cycles.)
    auto wait_acc = [&](int h = 0) {
      if (ew == 0) mbar_wait(acc_full(h), acc_phase[h]);
      acc_phase[h] ^= 1;
      epi_sync();
      tc_fence_after();
    };
    auto arrive_act = [&](int h = 0) { if (CG == 2) mbar_arrive_cluster(act_ready_leader[h]); else mbar_arrive(act_ready(h)); };
    // entry i of this step's walk -> board (search / self-play: the i-th game of my run that has a pending leaf)
    int32_t* my_list = dyn ? e.act_list + run_lo : nullptr;
    auto board_of = [&](int i) -> long long { i /= E; return dyn ? (long long)my_list[i] : run_lo + i; };
    // the form entry i (of board `board`) is evaluated in; 0 = identity
    auto form_of = [&](int i, long long board) -> int {
      if (a.form_mode == YY_FORM_FIXED) return a.form_fixed;
      if (a.form_mode == YY_FORM_AVERAGE) return form_at(i % E, g.n, g.m);
      if (a.form_mode == YY_FORM_HASHED) {
        const BB<NW> bb = load_bb<NW>(a.black, board, g.W) & geo.full, wb = load_bb<NW>(a.white, board, g.W) & geo.full;
        return hashed_form(stub_key(geo, bb, wb), a.form_seed, g.n, g.m);
      }
      return 0;
    };
    // One warp compacts the games of my run that have a pending leaf (from the front of my_list) and those still
    // selecting (from its back), and publishes both counts for step `iter_next` to every thread of the CTA (pair) --
    // read after the barrier in fetch_counts.
    auto compact = [&](int iter_next) {
      if (ew != 0) return;
      int n = 0, ns = 0;
      for (int base = 0; base < my_len; base += 32) {
        const int i = base + lane;
        const int np = i < my_len ? e.g_npending[run_lo + i] : 0;
        const unsigned m = __ballot_sync(kFull, np > 0), ms = __ballot_sync(kFull, np < 0);
        const unsigned below = (1u << lane) - 1u;
        if (np > 0) my_list[n + __popc(m & below)] = (int)(run_lo + i);
        if (np < 0) my_list[my_len - 1 - ns - __popc(ms & below)] = (int)(run_lo + i);
        n += __popc(m); ns += __popc(ms);
      }
      if (lane == 0) {
        volatile int* slot = cnt_s + (iter_next & 1) * 4 + rank * 2;
        slot[0] = n; slot[1] = ns;
        if (CG == 2) {
          const uint32_t peer = mapa_u32(smem_u32(const_cast<int*>(slot)), (uint32_t)(rank ^ 1));
          st_cluster_u32(peer, (uint32_t)n); st_cluster_u32(peer + 4, (uint32_t)ns);
        }
      }
    };
    if (dyn) {
      // self-play: slots without a search in progress (after a reset, or stopped on their move budget) get their next root;
      // arena: a slot whose model the turn flag names (set by the other half of the grid) roots its search
      if (a.mode >= YY_FUSED_SELFPLAY)
        for (int b = ew; b < my_len; b += TW_EPI_WARPS)
          if (e.g_npending[run_lo + b] == 0) advance_game<NW>(e, geo, (int)(run_lo + b), lane, a.mode);
      epi_sync();
      compact(0);
    }
    // a step without a tower pass (no game of the pair has a pending leaf): the epilogue warps advance the games that
    // are still selecting themselves
    auto run_selecting = [&]() {
      for (int k = ew; k < n_sel; k += TW_EPI_WARPS) {
        const int gi = my_list[my_len - 1 - k];
        const int np = tree_step_game<NW>(e, geo, gi, lane, nullptr, e.max_descents);
        if (np == 0 && a.mode >= YY_FUSED_SELFPLAY) advance_game<NW>(e, geo, gi, lane, a.mode);
      }
    };
    unsigned long long evals_here = 0;
    for (int iter = 0; iter < a.iterations; ++iter) {
      if (dyn) { fetch_counts(iter); if (!any_work) break; }
      evals_here += (unsigned long long)n_mine;
      for (int bb0 = 0; bb0 < n_struct; bb0 += a.batch_boards) {
        const int slim = batch_end(bb0);
        const int lim = slim < n_mine ? slim : n_mine;           // entries at or past `lim` are padding of the walk
        const int nbb = lim > bb0 ? lim - bb0 : 0;
        if (a.use_nn) {
          for (int b0 = bb0; b0 < slim; b0 += g.Gb) {
            const int T = tiles_for(b0, slim);
            const int T0 = half_split(T), nh = T0 < T ? 2 : 1;
            // The 4 warps that share a TMEM lane quarter split a half's tiles and, when the half has fewer than 4 tiles, the
            // 16-column chunks of a tile: with two tiles per half every (tile, quarter) has two warps, 4 chunks each.
            auto my_share = [&](int hh, int& t, int& c_lo, int& n_c) {
              const int tlo = hh ? T0 : 0, nt = (hh ? T : T0) - tlo;
              const int wpt = nt == 1 ? 4 : (nt == 2 ? 2 : 1);              // warps per (tile, quarter)
              t = tlo + sub4 / wpt;
              n_c = (TW_C / 16) / wpt;
              c_lo = (sub4 % wpt) * n_c;
              return t < tlo + nt;
            };
            // ---- stem input planes (board_to_input, neural_network.py:156-196) for my row of tile t ----
            auto stem_rows = [&](int t) {
              const int mi = t * 128 + quarter * 32 + lane;
              const int p = pos_p[mi];
              const int info = pos_tab[mi];
              uint4 c0 = make_uint4(0, 0, 0, 0);
              const int entry = b0 + (info >= 0 ? (info >> 8) : 0);
              if (info >= 0 && entry < lim) {
                const long long board = board_of(entry);
                const int cell = info & 255, y = cell / g.m, x = cell % g.m;
                const uint64_t* bb = a.black + board * g.W; const uint64_t* wb = a.white + board * g.W;
                // the network sees form f of the board: cell c reads cell form_src(f, c); fills are the transformed board's
                const int f = form_of(entry, board);
                auto bit = [&](const uint64_t* v, int c) { if (f) c = form_src(f, g.n, g.m, c); return (int)((v[c >> 6] >> (c & 63)) & 1ull); };
                const int isb = bit(bb, cell), isw = bit(wb, cell);
                int rc = 0, cc = 0;
                for (int xx = 0; xx < g.m; ++xx) { int c = y * g.m + xx; rc += bit(bb, c) | bit(wb, c); }
                for (int yy = 0; yy < g.n; ++yy) { int c = yy * g.m + x; cc += bit(bb, c) | bit(wb, c); }
                const float rf = (float)((double)rc / (double)g.m), cf = (float)((double)cc / (double)g.n);
                const float rf_hi = __bfloat162float(__float2bfloat16_rn(rf)), cf_hi = __bfloat162float(__float2bfloat16_rn(cf));
                // channels: 0 empty, 1 black, 2 white, 3 row fill, 4 col fill, 5/6 = bf16 residuals of 3/4 (same weights)
                c0.x = pack_bf16x2((isb | isw) ? 0.0f : 1.0f, isb ? 1.0f : 0.0f);
                c0.y = pack_bf16x2(isw ? 1.0f : 0.0f, rf_hi);
                c0.z = pack_bf16x2(cf_hi, rf - rf_hi);
                c0.w = pack_bf16x2(cf - cf_hi, 0.0f);
              }
              *reinterpret_cast<uint4*>(act + (size_t)(0 * TW_ROWS + TW_PAD + p) * 16) = c0;
              *reinterpret_cast<uint4*>(act + (size_t)(1 * TW_ROWS + TW_PAD + p) * 16) = make_uint4(0, 0, 0, 0);
            };
            // ---- one layer's epilogue for my row of tile t, 16-column chunks [c_lo, c_lo + n_c): accumulator -> bias, ReLU ->
            // bf16 activations in place (conv1 parks the skip input in TMEM first); head convolution -> head features in L2 ----
            auto layer_rows = [&](int l, int t, int c_lo, int n_c, const float* bias) {
              const bool is_head = (l == L - 1);
              const bool is_conv1 = (l >= 1 && l <= 2 * g.blocks && (l & 1) == 1);
              const int mi = t * 128 + quarter * 32 + lane;
              const int p = pos_p[mi];
              const int info = pos_tab[mi];
              const int entry = b0 + (info >= 0 ? (info >> 8) : 0);
              const bool real = info >= 0 && entry < lim;
              const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(t * 128);
              uint8_t* rowp = act + (size_t)(TW_PAD + p) * 16;
              if (!is_head) {
                // one 16-column chunk: bias + ReLU (+ park the skip input in TMEM) -> two 16-byte channel chunks in place
                auto process = [&](const uint32_t (&r)[16], int cc) {
                  uint4* d0 = reinterpret_cast<uint4*>(rowp + (size_t)(2 * cc) * TW_ROWS * 16);
                  uint4* d1 = reinterpret_cast<uint4*>(rowp + (size_t)(2 * cc + 1) * TW_ROWS * 16);
                  if (is_conv1) {  // skip connection: conv2 will accumulate on top of the block input
                    const uint4 x0 = *d0, x1 = *d1;
                    uint32_t xr[16];
                    const uint32_t xs[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
                    for (int q = 0; q < 8; ++q) { xr[2 * q] = xs[q] << 16; xr[2 * q + 1] = xs[q] & 0xffff0000u; }
                    tc_st16(taddr + cc * 16, xr);
                  }
                  const float4* b4 = reinterpret_cast<const float4*>(bias + cc * 16);
                  float v[16];
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    const float4 bq = b4[q];
                    v[4 * q + 0] = fmaxf(__uint_as_float(r[4 * q + 0]) + bq.x, 0.0f);
                    v[4 * q + 1] = fmaxf(__uint_as_float(r[4 * q + 1]) + bq.y, 0.0f);
                    v[4 * q + 2] = fmaxf(__uint_as_float(r[4 * q + 2]) + bq.z, 0.0f);
                    v[4 * q + 3] = fmaxf(__uint_as_float(r[4 * q + 3]) + bq.w, 0.0f);
                  }
                  if (!real) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = 0.0f;
                  }
                  *d0 = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
                  *d1 = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
                };
                // software pipeline: the TMEM load of chunk c+1 is in flight while chunk c is processed (n_c is even)
                uint32_t ra[16], rb[16];
                const int c_hi = c_lo + n_c;
                tc_ld16(taddr + c_lo * 16, ra);
#pragma unroll 1
                for (int cc = c_lo; cc < c_hi; cc += 2) {
                  tc_wait_ld();
                  tc_ld16(taddr + (cc + 1) * 16, rb);
                  process(ra, cc);
                  tc_wait_ld();
                  if (cc + 2 < c_hi) tc_ld16(taddr + (cc + 2) * 16, ra);
                  process(rb, cc + 1);
                }
                if (is_conv1) tc_wait_st();
              } else {
                __nv_bfloat16* dst = a.headfeat + (size_t)(run_lo * E + entry) * (TW_HEADC * g.A) + (info & 255);   // by walk entry
                const int h_n = n_c >= 2 ? n_c / 2 : 1, h_lo = n_c >= 2 ? c_lo / 2 : c_lo;   // 4 chunks of 16 head channels over the same warps
#pragma unroll 1
                for (int cc = h_lo; cc < h_lo + h_n && cc < TW_HEADC / 16; ++cc) {
                  uint32_t r[16];
                  tc_ld16(taddr + cc * 16, r);
                  tc_wait_ld();
                  if (real) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                      dst[(size_t)(cc * 16 + j) * g.A] = __float2bfloat16_rn(fmaxf(__uint_as_float(r[j]) + bias[cc * 16 + j], 0.0f));
                  }
                }
              }
            };

            if (skewed(T)) {
              // ---- skewed tiles: the 4 warps of tile `sub4` follow THEIR tile through the tower (per-tile barriers, per-tile bias
              // double buffer, one named barrier of 128 threads per layer); warps without a tile (T == 3) sit the group out ----
              const int t = sub4;
              if (t < T) {
                float* bias_t = reinterpret_cast<float*>(smem + SM_BIAS_T) + t * 2 * TW_C;
                const int tl = (ew & 3) * 32 + lane;                       // my index among the tile's 128 threads
                auto tile_sync = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(3 + t) : "memory"); };
                const uint32_t ready = CG == 2 ? mapa_u32(act_ready_t(t), 0) : act_ready_t(t);
                auto arrive_t = [&]() { if (CG == 2) mbar_arrive_cluster(ready); else mbar_arrive(ready); };
                stem_rows(t);
                bias_t[tl] = __ldg(wf(a.conv_bias) + tl);                      // stem biases (buffer 0)
                tc_fence_before();
                fence_proxy_async_smem();
                arrive_t();
                for (int l = 0; l < L; ++l) {
                  mbar_wait(acc_full_t(t), (acct_phase >> t) & 1u);
                  acct_phase ^= 1u << t;
                  tc_fence_after();
                  tile_sync();           // this layer's biases are staged by all four warps; the other buffer is free
                  if (l + 1 < L) bias_t[((l + 1) & 1) * TW_C + tl] = __ldg(wf(a.conv_bias) + (size_t)(l + 1) * TW_C + tl);
                  layer_rows(l, t, 0, TW_C / 16, bias_t + (l & 1) * TW_C);
                  tc_fence_before();
                  if (l + 1 < L) {
                    fence_proxy_async_smem();
                    arrive_t();
                  }
                }
              }
              continue;
            }

            for (int hh = 0; hh < nh; ++hh) {
              int t, c_lo, n_c;
              if (my_share(hh, t, c_lo, n_c) && c_lo == 0) stem_rows(t);
              tc_fence_before();
              fence_proxy_async_smem();
              arrive_act(hh);
            }
            if (etid < TW_C) bias_s[etid] = __ldg(wf(a.conv_bias) + etid);     // stem biases (buffer 0)

            for (int l = 0; l < L; ++l) {
              const bool is_head = (l == L - 1);
              // this layer's biases were staged in shared memory while its MMAs ran (an LDG per chunk sat on the
              // epilogue's critical path: 40 % of its stall samples); double buffered by layer parity
              const float* bias = bias_s + (l & 1) * TW_C;
              for (int hh = 0; hh < nh; ++hh) {
                wait_acc(hh);
                int t, c_lo, n_c;
                if (my_share(hh, t, c_lo, n_c)) layer_rows(l, t, c_lo, n_c, bias);
                tc_fence_before();
                if (!is_head) {
                  fence_proxy_async_smem();
                  arrive_act(hh);
                }
              }
              if (!is_head && etid < TW_C) bias_s[((l + 1) & 1) * TW_C + etid] = __ldg(wf(a.conv_bias) + (size_t)(l + 1) * TW_C + etid);
            }
          }

          // ---- FC heads for the batch: feature panels (global/L2 -> shared, K-major core matrices, boards = rows)
          epi_sync();   // every board's head features are written and visible CTA-wide
          phase(0);
          for (int q = 0; q < 2 * fc.n_panels; ++q) {
            const int h = q / fc.n_panels, p = q % fc.n_panels;
            if (q > 0) { wait_acc(); sub(6); }   // previous panel consumed
            const int nchunks = panel_stages(p) * 8;
            const int kbase = p * FC_PANEL_STAGES * 64;
            const __nv_bfloat16* src0 = a.headfeat + (size_t)(run_lo * E + bb0) * (TW_HEADC * g.A) + (size_t)h * fc.Kh + kbase;
            for (int idx = etid; idx < nbb * nchunks; idx += TW_EPI_THREADS) {
              const int b = idx / nchunks, j = idx - b * nchunks;
              const bool valid = kbase + j * 8 < fc.Kh;      // K padding up to the stage boundary must be zero
              cp_async16(act_base + (uint32_t)(j * FC_LBO + b * 16), src0 + (size_t)b * (TW_HEADC * g.A) + (valid ? j * 8 : 0), valid);
            }
            cp_async_commit();
            cp_async_wait<0>();
            tc_fence_before();
            fence_proxy_async_smem();
            arrive_act();
            sub(5);
          }
          wait_acc();
          sub(6);
          // D tiles -> scratch: policy logits (+bias), value hidden units relu(.+b1) * w2   (lane = output unit)
          if (tile0 < fc.Tp + 2) {
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(tile0 * FC_N * CG + rank * FC_N);
            uint32_t r0[16], r1[16];
            tc_ld16(taddr, r0);
            tc_ld16(taddr + 16, r1);
            tc_wait_ld();
            const int row = quarter * 32 + lane;
            if (tile0 < fc.Tp) {
              const int o = tile0 * 128 + row;
              if (o < g.A) {
                const float bo = __ldg(wf(a.fc_policy_b) + o);
#pragma unroll
                for (int b = 0; b < 16; ++b) { sc_logit[b * 256 + o] = __uint_as_float(r0[b]) + bo; sc_logit[(b + 16) * 256 + o] = __uint_as_float(r1[b]) + bo; }
              }
            } else {
              const int o = (tile0 - fc.Tp) * 128 + row;
              const float b1 = __ldg(wf(a.fc_value1_b) + o), w2 = __ldg(wf(a.fc_value2_w) + o);
#pragma unroll
              for (int b = 0; b < 16; ++b) {
                sc_hidden[b * 256 + o] = fmaxf(__uint_as_float(r0[b]) + b1, 0.0f) * w2;
                sc_hidden[(b + 16) * 256 + o] = fmaxf(__uint_as_float(r1[b]) + b1, 0.0f) * w2;
              }
            }
          }
          tc_fence_before();
          epi_sync();
          sub(7);
          phase(1);
        }

        // ---- per board: softmax over all A logits (predict, neural_network.py:152), value_fc2 + tanh (:121), tree step
        if (dyn && slim == n_struct && etid == 0) *(cnt_s + 8) = iter + 1;    // last tree phase of the step: background warps wind up
        // (one warp per board: its E entries are consecutive and in this batch, since E divides batch_boards)
        for (int b0e = ew * E; b0e < nbb; b0e += TW_EPI_WARPS * E) {
          const long long board = board_of(bb0 + b0e);
          if (a.use_nn) {
            float vsum = 0.0f;
            for (int q = 0; q < E; ++q) {
              const int b = b0e + q;
              const int f = form_of(bb0 + b, board);
              const float* lg = sc_logit + b * 256;
              float mx = -INFINITY;
              for (int k = lane; k < g.A; k += 32) mx = fmaxf(mx, lg[k]);
              for (int off = 16; off; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
              float sum = 0.0f;
              for (int k = lane; k < g.A; k += 32) sum += expf(lg[k] - mx);
              for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
              // output k of form f is the prior (logit) of action form_src(f, k); averaging: fp32 sum in ascending form
              // order, then / E (a power of two: exact)
              for (int k = lane; k < g.A; k += 32) {
                const long long o = board * g.A + (f ? form_src(f, g.n, g.m, k) : k);
                const float p = expf(lg[k] - mx) / sum;
                if (E == 1) {
                  a.policy[o] = p;
                  if (a.logits) a.logits[o] = lg[k];
                } else {
                  const float s = q ? a.policy[o] + p : p;
                  a.policy[o] = q + 1 == E ? s * (1.0f / (float)E) : s;
                }
              }
              float acc = 0.0f;
              for (int k = lane; k < 256; k += 32) acc += sc_hidden[b * 256 + k];
              for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
              const float v = tanhf(acc + __ldg(wf(a.fc_value2_b)));
              if (E == 1) { if (lane == 0) a.value[board] = v; }
              else vsum += v;
              __syncwarp();
            }
            if (E > 1 && lane == 0) a.value[board] = vsum * (1.0f / (float)E);
            __syncwarp();
          }
          if (dyn) {
            const int np = tree_step_game<NW>(e, geo, (int)board, lane, nullptr, e.max_descents);
            // search complete: the game makes its move and roots its next search now (self_play.py:139-190, :91-137)
            // (arena: the game makes its move and hands the turn to the other model's slot)
            if (np == 0 && a.mode >= YY_FUSED_SELFPLAY) advance_game<NW>(e, geo, (int)board, lane, a.mode);
          }
        }
        phase(2);
        if (a.use_nn) {
          epi_sync();     // scratch consumed, new leaves published
          phase(3);
          for (int i = etid; i < TW_CHUNKS * TW_ROWS; i += TW_EPI_THREADS) reinterpret_cast<uint4*>(act)[i] = make_uint4(0, 0, 0, 0);
          epi_sync();     // zero padding rows restored before the next stem writes its planes
          phase(4);
        }
      }
      if (n_struct == 0) run_selecting();
      if (dyn && iter + 1 < a.iterations) {
        tree_sync();      // every tree step of this CTA is done (epilogue and background warps)
        compact(iter + 1);
      }
    }
    if (dyn && etid == 0 && evals_here) atomicAdd(&e.stats->tower_evals, evals_here);
    if (a.dbg && lane == 0 && (blockIdx.x == 0 || blockIdx.x == 100))
      for (int k = 0; k < 8; ++k) a.dbg[600 + (blockIdx.x ? 160 : 0) + ew * 8 + k] = ph_acc[k];
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  if (a.dbg && tid == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); a.dbg[129 + 2 * blockIdx.x] = (long long)gt; }
  if (warp == 1) { if (CG == 2) tmem_dealloc2(tmem_base, 512); else tmem_dealloc(tmem_base, 512); }
}

// ------------------------------------------------------------------------------------------------ host side
template <int NW, int CG>
static int launch_fused(NNState& nn, const FusedArgs& fa, const EngineDev& dev, uint32_t rule_flags, int grid, cudaStream_t s) {
  static bool attr_set[8] = {};
  if (!attr_set[nn.device & 7]) {
    YY_CUDA_OK(cudaFuncSetAttribute(fused_kernel<NW, CG>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL));
    attr_set[nn.device & 7] = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(TW_THREADS); cfg.dynamicSmemBytes = SM_TOTAL; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const Geo<NW> geo = make_geo<NW>(nn.rows, nn.cols, rule_flags);
  YY_CUDA_OK(cudaLaunchKernelEx(&cfg, fused_kernel<NW, CG>, fa, dev, geo));
  YY_LAUNCH_CHECK();
  return YY_OK;
}

// Runs `iterations` evaluation (+ tree) steps over boards [0, count) in ONE launch.
//   dev == nullptr : plain forward (do_tree off); policy/value/logits are the caller's output arrays.
//   dev != nullptr : whole search over dev->leaf_* / eval_* (slot = game; leaves_per_step must be 1).
//   YY_FUSED_ARENA : boards [count/2, count) are evaluated with the image `weights_b` (same geometry as the loaded one).
int nn_fused_run(NNState& nn, const EngineDev* dev, uint32_t rule_flags, const uint64_t* black, const uint64_t* white, int64_t count,
                 float* policy, float* value, float* logits, int iterations, bool use_nn, int mode, const FormSpec& forms,
                 cudaStream_t s, const void* weights_b) {
  if (use_nn) {
    if (!nn.attrs_set) return set_error(YY_ERR_STATE, "engine was not created with the NN evaluator");
    if (!nn.weights) return set_error(YY_ERR_STATE, "no weights loaded (yy_engine_load_weights)");
  }
  if (forms.mode != YY_FORM_IDENTITY && !use_nn) return set_error(YY_ERR_INVALID, "symmetric evaluation needs the NN evaluator");
  if (forms.mode == YY_FORM_FIXED && !form_valid(forms.form, nn.rows, nn.cols))
    return set_error(YY_ERR_INVALID, "form %d is not a form of a %dx%d board", forms.form, nn.rows, nn.cols);
  if (forms.mode == YY_FORM_AVERAGE && logits) return set_error(YY_ERR_INVALID, "no logits when averaging over the forms");
  const int E = form_entries(forms.mode, nn.rows, nn.cols);
  if (count <= 0 || iterations <= 0) return YY_OK;
  if (count > nn.max_boards || count * E > nn.max_entries)
    return set_error(YY_ERR_INVALID, "fused run: %lld boards x %d forms exceed the head-feature scratch (%d boards, %d entries)",
                     (long long)count, E, nn.max_boards, nn.max_entries);
  if ((mode != YY_FUSED_FORWARD) != (dev != nullptr)) return set_error(YY_ERR_INVALID, "fused run: mode / engine state mismatch");
  const bool arena = mode == YY_FUSED_ARENA;
  if (arena && (!use_nn || !weights_b || (count & 1))) return set_error(YY_ERR_INVALID, "fused arena run: two images, an even count");
  FusedArgs fa{};
  fa.g = make_fused_geo(nn.rows, nn.cols, nn.blocks);
  fa.fc = make_fc_geo(nn.A);
  if (use_nn) {
    const WeightLayout wl = weight_layout(nn.rows, nn.cols, nn.blocks);
    const uint8_t* wimg = static_cast<const uint8_t*>(nn.weights);
    fa.conv_stream = wimg + wl.conv_stream_pair;     // stages split in two N halves, one per CTA of the pair
    fa.conv_bias = reinterpret_cast<const float*>(wimg + wl.conv_bias);
    fa.fc_stream = wimg + wl.fc_stream;
    fa.fc_policy_b = reinterpret_cast<const float*>(wimg + wl.fc_policy_b);
    fa.fc_value1_b = reinterpret_cast<const float*>(wimg + wl.fc_value1_b);
    fa.fc_value2_w = reinterpret_cast<const float*>(wimg + wl.fc_value2_w);
    fa.fc_value2_b = reinterpret_cast<const float*>(wimg + wl.fc_value2_b);
    fa.headfeat = reinterpret_cast<__nv_bfloat16*>(nn.scratch);
  }
  fa.black = black; fa.white = white; fa.count = count;
  fa.policy = policy; fa.value = value; fa.logits = logits;
  fa.iterations = iterations; fa.mode = mode; fa.use_nn = use_nn ? 1 : 0;
  fa.dbg = nn.dbg;
  fa.split_halves = nn.dbg_flags & 1;
  fa.no_skew = (nn.dbg_flags >> 1) & 1;
  fa.batch_boards = fused_batch_boards(fa.g);
  fa.form_mode = forms.mode; fa.form_fixed = forms.form; fa.form_seed = forms.seed; fa.n_avg = E;
  fa.batch_boards -= fa.batch_boards % E;   // a board's E entries share a heads pass (E in {1, 4, 8} <= every batch)
  // equal contiguous runs of boards per CTA (a search keeps its games on the same SM from the first to the last simulation)
  int sms = nn.num_sms > 0 ? nn.num_sms : 148;
  // (small batches -- an arena of 16 games, a search of a few hundred positions -- are spread over as many CTAs as there are boards
  // rather than packed into full groups: fewer tiles per CTA and step, i.e. lower latency, and the SMs would idle otherwise)
  long long per = (count + sms - 1) / sms;
  if (per < 1) per = 1;
  fa.boards_per_cta = (int)per;
  int grid = (int)((count + per - 1) / per);
  grid = (grid + 1) & ~1;                // whole CTA pairs; a trailing follower without boards only mirrors its leader's walk
  fa.half_grid = grid; fa.half_count = count;
  if (arena) {                           // each half of the grid gets whole CTA pairs over one model's boards
    const long long half = count / 2;
    per = (half + sms / 2 - 1) / (sms / 2);
    if (per < 1) per = 1;
    fa.boards_per_cta = (int)per;
    fa.half_grid = ((int)((half + per - 1) / per) + 1) & ~1;
    fa.half_count = half;
    fa.wb_off = (long long)((uintptr_t)weights_b - (uintptr_t)nn.weights);
    grid = 2 * fa.half_grid;
  }
  EngineDev d{};
  if (dev) d = *dev;
  if (nn.profiling) {
    if (nn.ev_used == nn.ev_cap) { int rc = nn_get_profile(nn, nullptr, nullptr, nullptr); if (rc) return rc; }
    YY_CUDA_OK(cudaEventRecord(nn.ev[2 * nn.ev_used], s));
  }
  int rc = YY_OK;
  YY_DISPATCH_NW(nn.A, rc = (launch_fused<NW, 2>(nn, fa, d, rule_flags, grid, s)));
  if (rc) return rc;
  if (nn.profiling) {
    YY_CUDA_OK(cudaEventRecord(nn.ev[2 * nn.ev_used + 1], s));
    ++nn.ev_used; ++nn.tower_launches; nn.tower_boards += count * iterations;   // upper bound; the executed number is Stats::tower_evals
  }
  return YY_OK;
}

}  // namespace yy
