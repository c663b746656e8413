/*
 * yinyang_b200.h -- C ABI of the B200-native Yin-Yang self-play engine.
 *
 * This is the drop-in boundary for the self-play hot path of
 * Arash-san/YinYang-Game-AlphaZero.  Every entry point names the reference
 * interface (file:line, relative to the upstream repository root) it replaces.
 * Plain pointers and sizes only; no torch / C++ types.  All `*_dev` pointers
 * are CUDA device pointers owned by the caller; `stream` is a cudaStream_t
 * passed as void* (NULL = legacy default stream).  Every function returns 0 on
 * success or a negative yy_status; yy_last_error() gives the message.  Nothing
 * here has a CPU fallback: without a CUDA device the compute calls fail.
 *
 * Board encoding ("bitboards"): cell (x, y) of an n x m board is action
 * a = x*m + y (yin_yang_game.py:180-186); bit (a & 63) of 64-bit word (a >> 6).
 * A board is W = ceil(n*m/64) words of black followed (in a separate array) by
 * W words of white; arrays are board-major: word w of board i at [i*W + w].
 * Supported: n, m <= 32 and n*m <= 256 (6x6, 8x8, 16x16 of BASELINE.json).
 * Players are +1 (black) / -1 (white) (yin_yang_logic.py:8-11).
 */
#ifndef YINYANG_B200_H
#define YINYANG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YY_ABI_VERSION 2

typedef enum {
  YY_OK = 0,
  YY_ERR_INVALID = -1,   /* bad argument / unsupported board size            */
  YY_ERR_CUDA = -2,      /* CUDA runtime error (message in yy_last_error)    */
  YY_ERR_NO_DEVICE = -3, /* no CUDA device: there is no CPU fallback         */
  YY_ERR_CAPACITY = -4,  /* a tree arena overflowed (raise edges_per_game)   */
  YY_ERR_STATE = -5      /* call sequence error (e.g. NN mode without weights) */
} yy_status;

/* rule_flags */
#define YY_RULE_ROWCOL 1u /* also ban completed single-colour rows/columns:
                             src/gui/static/js/yin_yang_game.js:338-384.  OFF
                             (default) == the Python rules used by self-play,
                             yin_yang_logic.py:31-56. */

/* Terminal codes written by yy_ended / yy_env_step (getGameEnded,
 * yin_yang_game.py:80-110): the host maps them to the reference's return
 * values 0 / +1 / -1 / 0.0001. */
#define YY_RESULT_ONGOING 0
#define YY_RESULT_WIN 1
#define YY_RESULT_LOSS (-1)
#define YY_RESULT_DRAW 2

int yy_abi_version(void);
const char *yy_last_error(void);
/* Number of CUDA devices visible (0 on a CPU-only box). */
int yy_device_count(void);
/* Kernels launched by this library in this process since load (bench.py's gpu_launches). */
int64_t yy_launch_count(void);

/* ------------------------------------------------------------------ rules --
 * Batched, stateless.  `count` boards; one thread per board. */

/* YinYangGame.getValidMoves (yin_yang_game.py:60-78) = YinYangLogic.get_valid_moves
 * (yin_yang_logic.py:111-120) over is_valid_move (:31-56): out_mask bit a = 1 iff
 * action a is legal for players[i]. */
int yy_legal_mask(int rows, int cols, uint32_t rule_flags, const uint64_t *black_dev, const uint64_t *white_dev,
                  const int8_t *players_dev, uint64_t *out_mask_dev, int64_t count, void *stream);

/* YinYangGame.getNextState (yin_yang_game.py:39-58) + place_piece (yin_yang_logic.py:24-29):
 * places players[i]'s piece at actions[i] if legal, otherwise leaves the board unchanged
 * (silent no-op); the turn passes either way.  In place. */
int yy_step(int rows, int cols, uint32_t rule_flags, uint64_t *black_dev, uint64_t *white_dev, int8_t *players_dev,
            const int32_t *actions_dev, int64_t count, void *stream);

/* YinYangGame.getGameEnded (yin_yang_game.py:80-110): YY_RESULT_* from players[i]'s perspective. */
int yy_ended(int rows, int cols, uint32_t rule_flags, const uint64_t *black_dev, const uint64_t *white_dev,
             const int8_t *players_dev, int8_t *out_result_dev, int64_t count, void *stream);

/* One environment step of BASELINE.md (getValidMoves + getNextState + getGameEnded fused):
 * out_mask = legal mask of the side to move BEFORE the action; boards/players updated in
 * place; out_result = YY_RESULT_* of the successor from the next player's perspective. */
int yy_env_step(int rows, int cols, uint32_t rule_flags, uint64_t *black_dev, uint64_t *white_dev,
                int8_t *players_dev, const int32_t *actions_dev, uint64_t *out_mask_dev, int8_t *out_result_dev,
                int64_t count, void *stream);

/* The reference's board arrays on the device: int8 [count][n*m] with 0 empty / +1 black / -1 white (YinYangLogic.board,
 * yin_yang_logic.py:14-22) -> bitboards, and back (out_boards) / a legal-move mask -> uint8 [count][n*m] of 0/1 (out_mask, the
 * layout of getValidMoves, yin_yang_game.py:60-78).  Either output of yy_unpack_boards may be NULL. */
int yy_pack_boards(int rows, int cols, const int8_t *boards_dev, uint64_t *black_dev, uint64_t *white_dev, int64_t count,
                   void *stream);
int yy_unpack_boards(int rows, int cols, const uint64_t *black_dev, const uint64_t *white_dev, const uint64_t *mask_dev,
                     int8_t *out_boards_dev, uint8_t *out_mask_dev, int64_t count, void *stream);

/* Synthetic-board generator of SURVEY 8d / BASELINE.json configs[1]: board i = empty board
 * advanced by plies[i] uniformly random legal plies (passes as in the rules), Philox stream
 * keyed by (seed, i).  Also the random-play opponent of evaluate mode (RandomPlayer.play,
 * yin_yang_players.py:14-42). */
int yy_random_playout(int rows, int cols, uint32_t rule_flags, uint64_t seed, const int32_t *plies_dev,
                      uint64_t *black_dev, uint64_t *white_dev, int8_t *players_dev, int64_t count, void *stream);

/* ----------------------------------------------------------------- engine --
 * Batched MCTS + evaluator + self-play driver for n_games concurrent games.
 * Replaces MCTS (src/yin_yang/ai/mcts.py:227-505) driven by SelfPlayWorker.play_game
 * (src/yin_yang/ai/self_play.py:72-192). */

typedef struct yy_engine yy_engine;

/* evaluator */
#define YY_EVAL_STUB 0 /* deterministic dyadic hash priors/values (parity mode)  */
#define YY_EVAL_NN 1   /* bf16 tcgen05 policy/value network (yy_engine_load_weights) */
#define YY_EVAL_EXTERNAL 2 /* caller fills priors/values between yy_search_* calls
                              (duck-typed neural_net.predict seam, mcts.py:295,394) */

/* mode_flags */
#define YY_MODE_SEARCH_AS_BLACK 1u /* self-play searches every position as player 1 and applies the move
                                      with the real player (self_play.py:99,135-137,163; SURVEY Q5).
                                      Default ON in the reference-compatible facade. */
#define YY_MODE_STEP_KERNELS 2u    /* run a search as one tree-step kernel launch (+ network launches) per
                                      simulation instead of ONE persistent kernel per search.  The persistent
                                      kernel (csrc/yy_fused.cu) is the default for the STUB and NN evaluators with
                                      leaves_per_step == 1; both produce identical trees. */
#define YY_MODE_EVAL_RANDOM_FORM 4u /* NN evaluator: evaluate every leaf in one dihedral form of the board (the order of
                                      augment_sample: identity, rot90 x1/x2/x3, flip left-right, flip up-down, transpose,
                                      anti-transpose; rectangular boards: forms 0, 2, 4, 5), chosen by a hash of the position
                                      and the engine seed: forms[mix64(stub_key(board) ^ seed) % F].  Same FLOPs as identity. */
#define YY_MODE_EVAL_AVERAGE_FORMS 8u /* NN evaluator: evaluate every leaf in all F forms (F = 8 square, 4 rectangular) and
                                      use the mean prior and value (fp32, ascending form order).  F x the network FLOPs and
                                      head-feature scratch.  Excludes YY_MODE_EVAL_RANDOM_FORM.  Both modes apply to searches,
                                      self-play and yy_evaluate; the STUB and EXTERNAL evaluators refuse them. */

typedef struct {
  int32_t rows, cols;
  int32_t n_games;          /* concurrent games (trees) on this GPU                       */
  int32_t n_sims;           /* num_simulations (mcts.py:231)                              */
  uint32_t rule_flags;
  uint32_t mode_flags;
  int32_t evaluator;        /* YY_EVAL_*                                                  */
  int32_t edges_per_game;   /* child-slot capacity per tree; 0 = worst case (n_sims+1)*A  */
  int32_t temperature_threshold; /* self_play.py:27 (10)                                  */
  int32_t replay_capacity;  /* self-play example ring (records)                           */
  int32_t nn_channels;      /* 128 (neural_network.py:39)                                 */
  int32_t nn_blocks;        /* 10                                                         */
  int32_t device;           /* CUDA device ordinal                                        */
  int32_t leaves_per_step;  /* K: leaves selected per game per step. 1 (default) = deterministic mode,
                               exact sequential MCTS; K>1 = throughput mode with virtual loss */
  float cpuct;              /* mcts.py:231 (default 1.0; weak-promoted to float32)        */
  int32_t descents_per_step; /* persistent kernel: simulations a game may start per evaluation step when they keep
                               ending in revisited terminals (no predict call, mcts.py:365-367); the search resumes in
                               the next step.  Bounds the latency one game adds to its CTA pair's step; the search result
                               does not depend on it.  0 = default (4); < 0 = unbounded */
  double dirichlet_alpha;   /* mcts.py:233 (0.3)                                          */
  double dirichlet_epsilon; /* mcts.py:233 (0.25; used in float64, mcts.py:309-311)       */
  uint64_t seed;            /* Philox key for noise / action sampling                     */
} yy_engine_config;

/* Bytes of device workspace the engine needs for cfg (caller allocates, 256-B aligned). */
int64_t yy_engine_workspace_bytes(const yy_engine_config *cfg);
/* Creates an engine over caller-owned device memory.  NULL on failure (see yy_last_error). */
yy_engine *yy_engine_create(const yy_engine_config *cfg, void *workspace_dev, int64_t workspace_bytes);
void yy_engine_destroy(yy_engine *e);

/* Bytes of the packed bf16 weight image for (rows, cols, channels, blocks); the image itself is
 * produced by the host-side packer (BN folded: neural_network.py:94-123 eval semantics) and
 * uploaded by the caller; the engine keeps the pointer.  Layout: csrc/yy_nn.cuh. */
int64_t yy_nn_weight_bytes(int rows, int cols, int channels, int blocks);
int yy_engine_load_weights(yy_engine *e, const void *weights_dev, int64_t bytes);
/* Section offsets of that image for the host-side packer: out[0..8] = conv_stream, conv_bias, fc_policy_w, fc_policy_b,
 * fc_value1_w, fc_value1_b, fc_value2_w, fc_value2_b, total bytes; out[9] = policy rows padded to 16; out[10], out[11] =
 * offset / bytes of the stage-ordered FC stream; out[12] = conv stream with N-halved stages (CTA-pair kernel).  13 values. */
int yy_nn_weight_layout(int rows, int cols, int channels, int blocks, int64_t *out);

/* MCTS.search (mcts.py:275-343) for all games at once.  Roots: one board per game.
 * noise_dev (may be NULL): float64 [n_games][A], one Dirichlet sample per legal root action in
 * ascending action order (mcts.py:298-312), mixed only for games with noise_mask_dev[g] != 0.
 * Runs root evaluation + n_sims simulations per game with the engine's evaluator and writes
 * root.get_children_visit_counts() (mcts.py:168-181) into out_counts_dev int32[n_games][A]. */
int yy_search(yy_engine *e, const uint64_t *root_black_dev, const uint64_t *root_white_dev,
              const int8_t *root_players_dev, const double *noise_dev, const uint8_t *noise_mask_dev,
              int32_t *out_counts_dev, void *stream);

/* External-evaluator stepping (YY_EVAL_EXTERNAL): yy_search_begin selects the root leaves;
 * the caller reads yy_engine_leaf_* (n_slots = n_games * leaves_per_step entries, slot = game*K + k), fills
 * priors float32[n_slots][A] (raw softmax entries, mcts.py:77-78) and values float32[n_slots], then calls
 * yy_search_advance, which expands +
 * backs up and selects the next leaves.  Returns in *out_active the number of games that
 * still need an evaluation (0 = search finished; then call yy_search_counts). */
int yy_search_begin(yy_engine *e, const uint64_t *root_black_dev, const uint64_t *root_white_dev,
                    const int8_t *root_players_dev, const double *noise_dev, const uint8_t *noise_mask_dev,
                    void *stream);
int yy_search_advance(yy_engine *e, const float *priors_dev, const float *values_dev, int32_t *out_active,
                      void *stream);
int yy_search_counts(yy_engine *e, int32_t *out_counts_dev, float *out_child_w_dev, void *stream);
/* The search trees themselves (Node, mcts.py:28-48), for callers that walk below the root (the reference returns the
 * root Node from MCTS.search).  Arrays are game-major: node j of game g at [g * max_nodes + j] (node 0 = root), edge slot k
 * of game g at [g * edges_cap + k].  A reference Node is split in two: its statistics live in its parent's edge slot
 * (visits = edge_N, value_sum = edge_W, prior = edge_P, action = edge_action), its state in a node record created when a
 * simulation first expands it.  The children of node j are the n_edges[j] consecutive edge slots from edge_base[j], in
 * ascending action order; edge_child_meta packs the child summary: bits [32,48) = child node id + 1 (0: not created yet),
 * [57,60) = flags (1 expanded, 2 terminal, 4 no legal move). */
typedef struct {
  int32_t max_nodes, edges_cap, W;
  const int32_t *n_nodes, *n_edges_used;             /* [n_games] nodes / edge slots in use */
  const uint64_t *node_black, *node_white;           /* [n_games * max_nodes * W] */
  const int32_t *node_edge_base; const int16_t *node_n_edges; const int8_t *node_player; const uint8_t *node_flags;
  const float *node_value;                           /* terminal value / cached value of a child-less node */
  const int32_t *edge_N; const float *edge_W; const float *edge_P; const uint64_t *edge_child_meta; const uint8_t *edge_action;
} yy_tree_view;
int yy_engine_tree_view(yy_engine *e, yy_tree_view *out);

/* Device pointers (owned by the engine) of the pending leaf batch: boards to evaluate and a
 * per-game flag (1 = needs evaluation). */
const uint64_t *yy_engine_leaf_black(yy_engine *e);
const uint64_t *yy_engine_leaf_white(yy_engine *e);
const uint8_t *yy_engine_leaf_active(yy_engine *e);

/* Runs the engine's evaluator once on `count` boards (batch inference entry point; replaces
 * YinYangNeuralNetwork.predict, neural_network.py:125-154, batched): out_policy float32[count][A]
 * = softmax over all A logits (no masking, :152), out_value float32[count], optional
 * out_logits float32[count][A]. */
int yy_evaluate(yy_engine *e, const uint64_t *black_dev, const uint64_t *white_dev, int64_t count,
                float *out_policy_dev, float *out_value_dev, float *out_logits_dev, void *stream);
/* yy_evaluate in a given dihedral form (NN evaluator only), whatever the engine's mode_flags.  form 0..7: the network
 * sees form `form` of every board (the form must keep the board's shape: rectangular boards take 0, 2, 4, 5) and its
 * outputs are mapped back, so out_policy / out_logits are indexed by the board's own actions.  form -1: the mean over
 * all forms of policy and value (no logits; needs a head-feature scratch of >= F boards: n_games x leaves_per_step >= F
 * or YY_MODE_EVAL_AVERAGE_FORMS). */
int yy_evaluate_form(yy_engine *e, const uint64_t *black_dev, const uint64_t *white_dev, int64_t count, int32_t form,
                     float *out_policy_dev, float *out_value_dev, float *out_logits_dev, void *stream);

/* Optional CUDA-event timing of the dominant kernel (the persistent search / forward kernel, csrc/yy_fused.cu),
 * recorded on the launching stream around every launch while enabled.  yy_engine_get_profile synchronises on the
 * recorded events and returns totals since profiling was enabled: launches, summed device milliseconds, leaf
 * evaluations (boards x simulations) those launches performed. */
int yy_engine_set_profiling(yy_engine *e, int enable);
int yy_engine_get_profile(yy_engine *e, int64_t *tower_launches, double *tower_ms, int64_t *tower_boards);
/* Developer tool: while dbg_dev != NULL (>= 1024 int64) the persistent kernel records per-CTA start / end
 * %globaltimer stamps at dbg_dev[128 + 2*cta ..] and, for CTAs 0 and 100, the cycles its epilogue warps spent in
 * each phase (tower, FC heads, softmax + tree step, barrier, re-zero, ...) at dbg_dev[600 ..] / [760 ..]. */
int yy_engine_set_debug_stamps(yy_engine *e, long long *dbg_dev);
/* Developer tool (A/B measurements in tools/): bit 0 = run the tower with the two halves of a group ping-ponging through the
 * tensor cores (epilogue hidden, weights streamed twice; slower in wall clock: profiles/r02_ab_pingpong_*.txt); bit 1 = the
 * tiles of a group in lock step through every layer as in round 1 instead of skewed (profiles/r02_ab_tile_*.txt). */
int yy_engine_set_debug_flags(yy_engine *e, int flags);

/* Self-play driver (SelfPlayWorker.play_game, self_play.py:72-192) for n_games game slots; a slot whose game ends
 * starts the next game from the empty board (generate_games, self_play.py:194-216).  One move = one full search +
 * action selection + state update; examples are appended to the replay ring.
 *
 * With the persistent search kernel (the default: STUB / NN evaluator, leaves_per_step 1) the games are ROLLING: one
 * launch plays them all, and a slot whose search is complete makes its move and roots its next search in the same
 * evaluation step, independently of the other slots -- a search that ends early (revisited terminal leaves need no
 * evaluation, mcts.py:365-367) never waits for the slowest search of the batch, and only games with a pending leaf
 * occupy tensor-core tiles.  Each game is still the exact sequential search of the reference.
 *   yy_selfplay_run      every slot makes exactly n_moves moves (the launch ends when the last slot has).
 *   yy_selfplay_advance  runs `iterations` evaluation steps (one leaf per game slot per step); searches in progress at
 *                        the end of the call continue in the next one.  Moves completed: yy_selfplay_get_stats.
 *   yy_selfplay_set_quota  at most total_games games are started since the last reset (< 0: unlimited); slots that
 *                        would need a game beyond the quota idle.  Game serial s is the same game whichever slot plays
 *                        it: all its random draws are keyed by (seed, s, ply).
 * yy_selfplay_run also works in the per-step-kernel modes (lock-step: prepare, search, move kernels per move). */
int yy_selfplay_reset(yy_engine *e, void *stream);
int yy_selfplay_run(yy_engine *e, int32_t n_moves, void *stream);
int yy_selfplay_advance(yy_engine *e, int64_t iterations, void *stream);
int yy_selfplay_set_quota(yy_engine *e, int64_t total_games);
/* Recorded random stream instead of the engine's Philox draws (parity seam: the reference draws from the global
 * np.random state -- np.random.choice, self_play.py:143-160; np.random.dirichlet, mcts.py:303-306):
 *   uniforms_dev float64[n_games][n_plies]  the uniform draw behind the action choice of game s at ply p: temperature 1 =
 *                the first action whose cumulative visit share exceeds u; temperature 0 = entry floor(u*k) of the k most
 *                visited actions in ascending order
 *   noise_dev    float64[n_games][A]        the Dirichlet sample mixed into the root priors of game s at ply 0, one
 *                value per legal action in ascending action order
 * Either may be NULL (= Philox).  Games / plies beyond the recorded range fall back to Philox.  The arrays stay owned
 * by the caller and must outlive the self-play calls. */
int yy_selfplay_set_random_stream(yy_engine *e, const double *uniforms_dev, const double *noise_dev, int32_t n_games,
                                  int32_t n_plies);
/* Playout cap randomisation of self-play (yy_selfplay_run / yy_selfplay_advance): each move is a full search (n_sims
 * simulations, noise as usual, recorded) with probability full_prob -- decided by a hash of (seed, game serial, ply) --
 * otherwise a fast search (fast_sims simulations, no noise, not recorded).  full_prob = 1 turns it off (the default).
 * Applies from the next search root each slot prepares; yy_search* ignore it.
 *   full(s, p) = (mix64(mix64(seed ^ 0x706c61796f757463) ^ ((uint64)(uint32)s << 20 | p)) >> 32) < llround(full_prob 2^32)
 * A fast move chooses, applies and ends the game exactly as a full one; it adds no replay record (stats: `moves`
 * counts every search, `examples` the full ones).  YY_ERR_INVALID for full_prob outside [0, 1] or NaN and for fast_sims
 * outside [1, n_sims]; YY_ERR_STATE with the EXTERNAL evaluator. */
int yy_selfplay_set_playout_cap(yy_engine *e, double full_prob, int32_t fast_sims);

typedef struct {
  int64_t moves;          /* searches completed                         */
  int64_t evals;          /* leaf evaluations requested                 */
  int64_t games_finished;
  int64_t examples;       /* records appended to the replay ring        */
  int64_t sims;           /* simulations completed                      */
  int32_t overflow;       /* non-zero if a tree arena overflowed        */
  int32_t max_depth;
  int64_t tower_evals;    /* boards evaluated by the persistent kernel (each a pending leaf or root) */
} yy_selfplay_stats;
int yy_selfplay_get_stats(yy_engine *e, yy_selfplay_stats *out, void *stream);
/* Device address of the live counters: 7 x int64 = moves, evals, games_finished, examples, sims, (overflow | max_depth << 32),
 * tower_evals.  For stream-ordered snapshots (copy it after a self-play launch, on the same stream) without a
 * synchronisation: e.g. to drain the records of step k while step k + 1 runs. */
const void *yy_selfplay_stats_dev(yy_engine *e);

/* Replay record i (i < min(examples, replay_capacity)), struct-of-arrays on the device:
 *   black/white  uint64[cap][W]   position before the move (self_play.py:140)
 *   counts       uint16[cap][A]   root visit counts; pi = counts / sum in float64 (mcts.py:209)
 *   game_serial  int32[cap]       index into the results table
 *   ply          int16[cap], player int8[cap]
 * results: int8[results_capacity] YY_RESULT_* of game serial s at [s % results_capacity], from the perspective the
 * reference assigns to every example of that game (self_play.py:170-181; SURVEY Q6). */
typedef struct {
  const uint64_t *black, *white;
  const uint16_t *counts;
  const int32_t *game_serial;
  const int16_t *ply;
  const int8_t *player;
  const int8_t *results;
  int32_t results_capacity;
} yy_replay_view;
int yy_selfplay_replay(yy_engine *e, yy_replay_view *out);

/* Current live boards of the n_games slots (device pointers owned by the engine). */
const uint64_t *yy_engine_game_black(yy_engine *e);
const uint64_t *yy_engine_game_white(yy_engine *e);
const int8_t *yy_engine_game_player(yy_engine *e);

/* ---------------------------------------------------------------------------------------------
 * Replay records -> training tensors (SURVEY 8f-1).  Replaces create_dataset_from_games /
 * DataProcessor.preprocess_sample / augment_sample (src/yin_yang/ai/data_utils.py:16-215) over
 * board_to_input (neural_network.py:156-196) for a whole replay buffer at once.  Per record r the 8 forms of
 * augment_sample, in its order (identity, rot90 x1/x2/x3, flip left-right, flip up-down, transpose,
 * anti-transpose), sample index 8r + form:
 *   out_planes float32[8*count][5][n][m], out_policy float32[8*count][A], out_values float32[8*count] (optional).
 * Policy source: counts uint16[count][A] (visit counts: policy = counts / sum in float64, uniform when the sum
 * is 0 -- Node.get_children_distribution at temperature 1, mcts.py:183-215 -- rounded to float32 like
 * torch.FloatTensor(policy), data_utils.py:34) or, when counts is NULL, policy float32[count][A] as is.
 * Square boards only (the reference rotates by 90 degrees).  Bit-exact against the reference. */
int yy_augment_samples(int rows, int cols, const uint64_t *black_dev, const uint64_t *white_dev,
                       const uint16_t *counts_dev, const float *policy_dev, const float *values_dev, int64_t count,
                       float *out_planes_dev, float *out_policy_dev, float *out_values_dev, void *stream);

/* The same without augmentation (DataProcessor.preprocess_sample for a whole buffer, data_utils.py:16-37;
 * create_dataset_from_games(..., augment=False)): out_planes float32[count][5][n][m], out_policy float32[count][A],
 * out_values float32[count] (optional).  Any supported board shape. */
int yy_dataset_samples(int rows, int cols, const uint64_t *black_dev, const uint64_t *white_dev,
                       const uint16_t *counts_dev, const float *policy_dev, const float *values_dev, int64_t count,
                       float *out_planes_dev, float *out_policy_dev, float *out_values_dev, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Learner-step primitives (SURVEY 8f-2).  Together they replace one optimisation step of
 * AlphaZeroTrainer.train (src/yin_yang/ai/trainer.py:67-161): YinYangNeuralNetwork.forward in training mode
 * (neural_network.py:94-123; nn.BatchNorm2d batch statistics), CrossEntropyLoss(soft targets) + MSELoss
 * (trainer.py:60-61,131-133), backward, and torch.optim.Adam(lr, weight_decay) (trainer.py:52-56,136-137).
 * The host side (yinyang-game-alphazero_b200/learner.py) strings them into the layer sequence and captures the
 * step in one CUDA graph.  Activations are float32 [positions][channels] (positions = batch x cells, NHWC);
 * every matrix is row-major with a leading dimension in floats; all pointers are device pointers. */

/* C[M,N] = [C +] A[M,K] * B[N,K]^T (+ bias[n]) (ReLU) on the tensor cores (tcgen05.mma kind::tf32, fp32 accumulate in
 * TMEM) -- nn.Conv2d / nn.Linear forward (neural_network.py:94-123) and both of their gradients.
 *   a_mode YY_OP_K        A is [M][K] row-major (lda)
 *          YY_OP_K_CONV   implicit im2col: A[p][t*cin + ci] = X[p + d(t)][ci], X = [positions][cin] (lda), zero outside
 *                         the board; t = kh*3 + kw of nn.Conv2d(kernel_size=3, padding=1); conv->flip mirrors the taps
 *                         (the gather of the backward-data pass)
 *   b_mode YY_OP_K        B is [N][K] row-major (ldb)
 *          YY_OP_K_CONVT  implicit transposed im2col: B[t*cin + ci][p] = XT[ci][p + d(t)], XT = [cin][positions] (ldb) --
 *                         the weight gradient of a 3x3 convolution, dW = dY^T * im2col(X), whose reduction index is the
 *                         position (K = positions, at most 8192 per K slice)
 * precision: YY_GEMM_3XTF32 splits every operand into the 19 bits a TF32 multiplier reads and the remainder and runs
 * three MMAs per K-slice (lo*hi + hi*lo + hi*hi): fp32-level results, what the fp32 reference computes; YY_GEMM_TF32 is
 * the single-pass variant (torch's default for fp32 convolutions on a GPU).  accumulate != 0: the product is added to C
 * (a skip connection's share of a gradient).  tile_n: output columns per CTA (16..128, multiple of 16); split_k >= 1
 * slices K over gridDim.z: the partial tiles of up to 8 consecutive slices are summed on chip by a thread-block cluster
 * (distributed shared memory, rank order); with more slices the clusters' sums go to ws (>= (split/cluster)*M*N floats)
 * and a reducer adds them in order, so results are bit-reproducible.  bn_sums (optional, float64 [2N], zero on entry, N dividing 128): receives the per-column
 * sum / sum of squares of the finished C, i.e. the statistics of the batch norm that follows (yy_lrn_bn_forward with
 * have_sums = 1 then skips its own pass).  lda/ldb/ldc/N/K multiples of 4, pointers 16-byte aligned. */
#define YY_GEMM_TF32 0
#define YY_GEMM_3XTF32 1
#define YY_OP_K 0
#define YY_OP_K_CONV 1
#define YY_OP_K_CONVT 2
typedef struct {
  double *sums;             /* float64 [2N], zero on entry                                    */
  const float *out;         /* NULL: forward statistics; else the layer's output (ReLU mask)  */
  int32_t ldo;
  const float *y;           /* the layer's batch-norm input                                   */
  int32_t ldy;
  const float *mean_invstd; /* float [2N] written by yy_lrn_bn_forward                        */
} yy_gemm_stats;
typedef struct {
  int32_t rows, cols; /* board */
  int32_t cin;        /* channels of the gathered activation tensor (multiple of 4) */
  int32_t flip;       /* mirror the taps                                            */
} yy_conv_geom;
int yy_lrn_gemm(const float *A, int lda, int a_mode, const float *B, int ldb, int b_mode, float *C, int ldc, int M, int N, int K,
                const float *bias, int relu, int accumulate, int tile_n, int split_k, float *ws, int64_t ws_floats,
                int precision, const yy_conv_geom *conv, const yy_gemm_stats *stats, const void *b_packed, void *stream);
/* The weights of `layers` layers ([128][K] row-major; layer l at base + offsets_dev[l], or base + l*layer_stride when
 * offsets_dev is NULL) -> out + l*yy_lrn_pack_b_bytes(128, K): per K stage of 32 the hi and lo operand tiles of the 3xTF32
 * GEMM in its shared-memory layout.  Once per optimisation step for the whole tower. */
int yy_lrn_pack_b(const float *base, const long long *offsets_dev, int64_t layer_stride, int layers, int N, int K, void *out,
                  void *stream);
int64_t yy_lrn_pack_b_bytes(int N, int K);
/* Developer tool: while dbg_dev != NULL (>= 128 int64) CTA (0,0,0) of every yy_lrn_gemm launch records clock64 stamps:
 * [0] start, [1] after setup, [4+6k .. 8+6k] producer phases of K-iteration k (start, slot free, copies issued, copies of
 * iteration k-1 landed, iteration k-1 split + published), [2] loop end, [119] accumulator complete, [3] epilogue end. */
int yy_lrn_gemm_debug_stamps(long long *dbg_dev);
/* out[c][r] = in[r][c] for `batch` matrices `in_stride` / `out_stride` floats apart (batch = 1: strides ignored). */
int yy_lrn_transpose(const float *in, int ldi, float *out, int ldo, int R, int C, int batch, int64_t in_stride,
                     int64_t out_stride, void *stream);
/* colT[t*C + c][p] = X[p + d(t)][c], zero outside the board: the transposed im2col the weight gradient of a 3x3
 * convolution reads (dW = dY^T * colT^T; the reduction index is the position). */
int yy_lrn_im2col_t(const float *X, int ldx, float *colT, int ldo, int64_t positions, int rows, int cols, int C,
                    void *stream);
/* Wt[l][ci][t*Cout + co] = W_l[co][t*Cin + ci], W_l = params + offsets_dev[l] (offsets NULL: one layer at params): the B
 * operands of the backward-data GEMMs of `layers` 3x3 convolutions of the same shape, in one launch. */
int yy_lrn_conv_weight_t(const float *params, const long long *offsets_dev, int layers, float *Wt, int Cout, int Cin,
                         void *stream);
/* planes float32 [boards][5][cells] (board_to_input, neural_network.py:156-196) -> X0 float32 [boards*cells][8]. */
int yy_lrn_planes_nhwc(const float *planes, float *X0, int64_t boards, int cells, void *stream);
/* out[c] = sum_r X[r][c] (bias gradients). */
int yy_lrn_colsum(const float *X, int ld, int R, int C, float *out, void *stream);
/* nn.BatchNorm2d in train() (neural_network.py:22-25,44): out = [relu](gamma*(Y-mean)*invstd + beta [+ residual]) with
 * the batch's own mean / biased variance over the P positions; writes mean_invstd float[2C] for the backward pass and
 * updates running_mean / running_var (unbiased variance, `momentum`) in place when not NULL.  sums_ws: float64[2C], ZERO
 * on entry (the host side zeroes one slot per layer and pass with a single memset per step), or -- have_sums != 0 --
 * already holding the column sums / sums of squares of Y (yy_lrn_gemm's bn_sums). */
int yy_lrn_bn_forward(const float *Y, int ld, int P, int C, const float *gamma, const float *beta,
                      const float *residual, int ldr, float *out, int ldo, int relu, float eps, float momentum,
                      double *sums_ws, int have_sums, float *mean_invstd, float *running_mean, float *running_var,
                      void *stream);
/* Backward of the above (and of the ReLU after it when Out != NULL: dZ = dOut*[Out > 0]):
 * dY = gamma*invstd*(dZ - mean(dZ) - xhat*mean(dZ*xhat)); dRes (optional) = dZ; dgamma = sum dZ*xhat; dbeta = sum dZ;
 * dbias (optional, zero on entry) += column sums of dY = the bias gradient of the convolution feeding this batch norm.
 * dYT (optional): also the transposed copy dYT[c][p] = dY[p][c] (ldt) the weight-gradient GEMM reads.
 * sums_ws: float64[2C], zero on entry, or -- have_sums != 0 -- already holding sum dZ*xhat / sum dZ (yy_lrn_gemm's stats). */
int yy_lrn_bn_backward(const float *dOut, int ldd, const float *Out, int ldo, const float *Y, int ldy, int P, int C,
                       const float *mean_invstd, const float *gamma, double *sums_ws, float *dY, int lddy,
                       float *dRes, int lddr, float *dgamma, float *dbeta, float *dbias, float *dYT, int ldt,
                       int have_sums, void *stream);
/* Both losses and their gradients at the heads (trainer.py:131-133; value head tail neural_network.py:119-121):
 * losses[0] = CrossEntropyLoss(logits, pi) with probability targets, losses[1] = MSELoss(tanh(relu(h).w2 + b2), z),
 * h = value_fc1's output before its ReLU; dlogits, dh (through that ReLU), dpre[B], v_out[B], dw2[H], db2[1]. */
int yy_lrn_heads_loss(const float *logits, int ldl, const float *pi, int A, const float *h, int ldh, int H,
                      const float *w2, const float *b2, const float *z, int B, float *dlogits, int lddl, float *dh,
                      int lddh, float *dpre, float *v_out, float *dw2, float *db2, float *losses, void *stream);
/* torch.optim.Adam step (L2 weight decay folded into the gradient) over one flat parameter buffer (n a multiple of 4).
 * step_state: 4 x int32 on the device; [0] = step counter (incremented first), [2..3] scratch for the bias corrections. */
int yy_lrn_adam(float *params, const float *grads, float *m, float *v, int64_t n, float lr, float beta1, float beta2,
                float eps, float weight_decay, int *step_state, void *stream);

/* tcgen05 self-test used by tests/ (C = A[M,K] * B[N,K]^T, bf16 in / fp32 out, operands in the
 * same no-swizzle K-major core-matrix layout the tower kernel uses).  Layout: csrc/yy_probe.cu. */
int yy_probe_umma(const void *a_dev, const void *b_dev, float *c_dev, int M, int N, int K, int a_row_offset,
                  int swap_lbo_sbo, void *stream);

/* Developer tool: kind::tf32 MMA with a TRANSPOSED ("MN-major") A operand staged in the canonical layout of a swizzle mode
 * (variant 0 none, 1 SWIZZLE_128B, 2 the same bytes declared SWIZZLE_128B_BASE32B); B K-major.  At [K][128], B [N][K], C [128][N].
 * Layout: csrc/yy_probe.cu. */
int yy_probe_tf32_mn(const float *at_dev, const float *b_dev, float *c_dev, int N, int K, int variant, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* YINYANG_B200_H */
