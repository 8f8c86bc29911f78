/*
 * oz_b200.h — C ABI of the B200-native OthelloZero self-play engine.
 *
 * Drop-in boundary for the reference's (Galtvam/OthelloZero) Python hot path; the
 * reference has no FFI of its own (SURVEY §8b), so every entry point cites the Python
 * interface it replaces (paths relative to the reference root).  Plain pointers and
 * sizes only; no torch types.  Every function returns 0 on success or a negative
 * OZ_ERR_* code; oz_last_error() returns a thread-local message.
 *
 * Conventions
 *   - A board is two uint64 bitboards, bit index r*8+c for every board size N in {4,6,8}
 *     (N<8 lives in the top-left corner).  "black/white" = reference channels 0/1
 *     (Othello/__init__.py:22-25); "own/opp" = canonical form, side to move first
 *     (othelo_mcts.py:24-25).  player: 0 = BLACK, 1 = WHITE.
 *   - Squares/actions are bit indices r*8+c (NOT r*N+c).
 *   - *_host functions take HOST buffers and do the H2D/D2H copies themselves (the call a
 *     user of the reference makes); *_dev functions take DEVICE pointers that are resident
 *     in HBM and a cudaStream_t passed as void*.
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails
 *     with OZ_ERR_CUDA.
 *   - Rules.  By default every move is played with the reference's flip rule: a move also flips
 *     opponent discs that lie beyond the bracketing own disc (Othello/__init__.py:216-235 has no
 *     `break`).  OR-ing OZ_RULES_STANDARD into a board_size argument selects standard Othello
 *     flipping (a run flips only up to the first own disc) for oz_rules_apply_*,
 *     oz_perft_playouts_* and oz_engine_config.board_size (search and self-play).  Legal moves, the
 *     initial position, the automatic pass, the terminal test and the scoring are the same under
 *     both rule sets; oz_rules_legal_moves_* and oz_net_blob_floats accept the flag and ignore it,
 *     so one value can be passed everywhere.
 *   - Scoring.  By default a finished game with equal disc counts counts as a BLACK win (the
 *     reference's max() over {BLACK, WHITE}, Othello/__init__.py:254-256).  OR-ing
 *     OZ_SCORING_STANDARD into oz_engine_config.board_size scores it as a draw, independently of the
 *     rule set: the search backs a drawn terminal up as the integer 0, and self-play records winner
 *     OZ_WINNER_DRAW.  Empty squares left over are not counted.  oz_rules_legal_moves_*,
 *     oz_rules_apply_*, oz_perft_playouts_* and oz_net_blob_floats accept the flag and ignore it
 *     (nothing they compute depends on the scoring).  Any other bit above the size is
 *     OZ_ERR_INVALID.
 *   - Passes and perft.  A side with no legal move passes automatically inside the move that left
 *     it without one: a pass is not a move of its own and does not use up a ply.  A full-tree perft
 *     counted with these calls therefore treats a finished game as a leaf and a pass as free, e.g.
 *     8x8 depths 1-9 under standard rules: 4, 12, 56, 244, 1396, 8200, 55092, 390216, 3005320
 *     (reference rules first differ at depth 7: 55032, 389164, 2994476).
 */
#ifndef OZ_B200_H
#define OZ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OZ_OK 0
#define OZ_ERR_INVALID (-1) /* bad argument (reference: AssertionError / TypeError) */
#define OZ_ERR_CUDA (-2)    /* CUDA runtime/driver failure, or no device */
#define OZ_ERR_NOMEM (-3)   /* device allocation failed / node pool exhausted */
#define OZ_ERR_STATE (-4)   /* call sequence error (reference: RuntimeError) */

#define OZ_ABI_VERSION 1

/* OR-ed into a board_size argument: standard Othello flipping instead of the reference's (see Conventions) */
#define OZ_RULES_STANDARD 0x100
/* OR-ed into a board_size argument: a finished game with equal disc counts is a draw, not a BLACK win (see Conventions).
 * 0x200 is not used: it stays OZ_ERR_INVALID everywhere. */
#define OZ_SCORING_STANDARD 0x400
/* self-play winner code of a drawn game under OZ_SCORING_STANDARD (oz_selfplay_get_records) */
#define OZ_WINNER_DRAW 2

/* flags returned by oz_rules_apply_* (one uint32 per position) */
#define OZ_MOVE_SWAPPED 1u  /* opponent moves next; outputs are in HIS frame (own/opp swapped) */
#define OZ_MOVE_PASSED 2u   /* opponent has no move, mover moves again (Othello/__init__.py:151-159) */
#define OZ_MOVE_FINISHED 4u /* neither side can move (Othello/__init__.py:249-252) */

/* prior sources for the search */
#define OZ_PRIOR_HASH 0 /* closed-form hash prior evaluated on device (SURVEY App. B.3) — parity/roofline mode */
#define OZ_PRIOR_HOST 1 /* leaves handed to the host, priors fed back (any object with .predict) */
#define OZ_PRIOR_NET 2  /* OthelloNNet bf16 tcgen05 tower on device */

/* per-game status (oz_search_get_status) */
#define OZ_GAME_IDLE 0      /* sims for the current root done / not started */
#define OZ_GAME_ACTIVE 1    /* simulations in progress */
#define OZ_GAME_WAIT_LEAF 2 /* waiting for priors of its pending leaf */
#define OZ_GAME_FINISHED 3  /* self-play game over */
#define OZ_GAME_POOL_FULL 4 /* node pool exhausted (error) */

typedef struct oz_engine oz_engine;

typedef struct oz_engine_config {
    int32_t device;          /* CUDA ordinal */
    int32_t board_size;      /* 4, 6 or 8 (Othello/__init__.py:29-36; the net needs 6 or 8), | OZ_RULES_STANDARD for
                                standard flipping in simulations and self-play moves, | OZ_SCORING_STANDARD for drawn
                                games scored as draws in the search and in self-play winners */
    int32_t max_games;       /* concurrent game slots (one warp each) */
    int32_t nodes_per_game;  /* node-pool capacity per game; reference keeps every node of an episode
                                (training.py:32), i.e. <= sims * plies */
    int32_t prior_mode;      /* OZ_PRIOR_* */
    int32_t log_visits;      /* keep per-move root visit counts of self-play games (tests) */
    int32_t eval_cache_log2; /* OZ_PRIOR_NET: log2(entries) of the cross-game evaluation cache (272 B/entry); 0 = off.
                                Identical positions are evaluated once; results are unchanged. */
    int32_t vl_width;        /* > 1: up to vl_width simulations of a game in flight per step (virtual loss); visit counts
                                then differ from the sequential reference by design. 0/1 = sequential, bit-exact. */
    double c_puct;           /* degree_exploration (MCTS/__init__.py:27,168-170) */
    uint64_t seed;           /* engine RNG seed (epsilon-greedy, synthetic starts) */
} oz_engine_config;

const char* oz_last_error(void);
int oz_abi_version(void);
int oz_device_count(int32_t* count);

/* ---- rules: Othello/__init__.py (stateless, batched) ------------------------------------ */
/* get_player_valid_actions (:208-214) as a mask per position. */
int oz_rules_legal_moves_host(int32_t device, int32_t board_size, const uint64_t* own, const uint64_t* opp,
                              uint64_t* moves, int64_t n);
int oz_rules_legal_moves_dev(int32_t board_size, const uint64_t* own, const uint64_t* opp, uint64_t* moves, int64_t n,
                             void* stream);
/* flip_board_squares (:237-247) + the turn logic of OthelloGame.play (:147-159) /
 * OthelloMCTS.get_next_state (othelo_mcts.py:43-49).  sq[i] must be a legal move, else flags[i]=0x80000000.
 * Outputs are in the frame of the side that moves next; next_legal may be NULL. */
int oz_rules_apply_host(int32_t device, int32_t board_size, const uint64_t* own, const uint64_t* opp,
                        const int32_t* sq, uint64_t* own_out, uint64_t* opp_out, uint32_t* flags,
                        uint64_t* next_legal, int64_t n);
int oz_rules_apply_dev(int32_t board_size, const uint64_t* own, const uint64_t* opp, const int32_t* sq,
                       uint64_t* own_out, uint64_t* opp_out, uint32_t* flags, uint64_t* next_legal, int64_t n,
                       void* stream);

/* get_board_players_points (:258-260): disc counts per colour; the winner is BLACK iff black_points >= white_points
 * (max() over the dict in BLACK, WHITE order, :254-256). */
int oz_rules_score_host(int32_t device, const uint64_t* black, const uint64_t* white, int32_t* black_points,
                        int32_t* white_points, int64_t n);
int oz_rules_score_dev(const uint64_t* black, const uint64_t* white, int32_t* black_points, int32_t* white_points,
                       int64_t n, void* stream);

/* ---- perft / random playouts: RandomOthelloAgent loop, agents.py:20-24,71-84 ------------- */
/* Game g (global id first_game_id+g) starts at initial_board(board_size) and plays
 * legal[mulhi32(sm64(sm64(sm64(seed) + id) + p) >> 32, popcount(legal))] at move index p (ascending bit order ==
 * row-major), with auto-pass/terminal as OthelloGame.play, for at most max_moves moves (<0: to the end).
 * info[g] = plies | player<<8 | finished<<9 | passes<<16.  moves (optional) = [n_games][64] squares, 0xFF padded. */
int oz_perft_playouts_host(int32_t device, int32_t board_size, uint64_t seed, uint64_t first_game_id,
                           int64_t n_games, int32_t max_moves, uint64_t* black, uint64_t* white, uint32_t* info,
                           uint8_t* moves);
int oz_perft_playouts_dev(int32_t board_size, uint64_t seed, uint64_t first_game_id, int64_t n_games,
                          int32_t max_moves, uint64_t* black, uint64_t* white, uint32_t* info, uint8_t* moves,
                          void* stream);

/* ---- exact endgame solver (stateless, batched) -------------------------------------------- */
#define OZ_SOLVE_MAX_EMPTIES 20
#define OZ_SOLVE_NONE (-128) /* move_margin: not a legal move; margin: position not searched (_dev only) */
/* Exact final disc margin own-opp (empties not counted) under perfect play, side to move = own.  The game is the
 * engine's: a side without a legal move passes, a position where neither side can move is finished and worth its disc
 * difference.  The margin does not depend on the scoring; the outcome under either scoring follows from its sign and
 * the mover's colour.
 * board_size as everywhere (| OZ_RULES_STANDARD selects the flip rule; OZ_SCORING_STANDARD accepted and ignored).
 * margin [n]; move_margin [n][64] by square bit, may be NULL (then one work item per position; else one per legal root
 * move, each searched with the full window, and margin = the row's maximum); a finished position, or one whose mover
 * must pass, has an all-OZ_SOLVE_NONE row.  nodes [n] (positions visited per position, may be NULL).
 * max_empties in [0, OZ_SOLVE_MAX_EMPTIES].  _host checks every position before launching (discs must not overlap, must
 * lie on the N x N board, at most max_empties empties) and fails with OZ_ERR_INVALID naming the first bad one; _dev does
 * not validate content and marks a position with more than max_empties empties OZ_SOLVE_NONE without searching it
 * (it allocates its scratch stream-ordered on `stream`). */
int oz_endgame_solve_host(int32_t device, int32_t board_size, const uint64_t* own, const uint64_t* opp, int64_t n,
                          int32_t max_empties, int8_t* margin, int8_t* move_margin, uint64_t* nodes);
int oz_endgame_solve_dev(int32_t board_size, const uint64_t* own, const uint64_t* opp, int64_t n,
                         int32_t max_empties, int8_t* margin, int8_t* move_margin, uint64_t* nodes, void* stream);

/* ---- engine ----------------------------------------------------------------------------- */
int oz_engine_create(const oz_engine_config* cfg, oz_engine** out);
int oz_engine_destroy(oz_engine* e);
int oz_engine_sync(oz_engine* e);
/* The engine's CUDA stream (cudaStream_t) for callers that enqueue their own work around it. */
void* oz_engine_stream(oz_engine* e);

/* ---- search: OthelloMCTS (othelo_mcts.py:9-88 over MCTS/__init__.py:19-187) --------------- */
/* OthelloMCTS.__init__ for n_games trees: clears node pools, sets roots.  black/white/player HOST arrays
 * (NULL = initial position, BLACK to move). game_ids (NULL = 0..n-1) key the per-game RNG streams. */
int oz_search_reset(oz_engine* e, int32_t n_games, const uint64_t* black, const uint64_t* white,
                    const int32_t* player, const uint64_t* game_ids);
/* Move roots without clearing trees (state argument of OthelloMCTS.simulate, othelo_mcts.py:22-26). */
int oz_search_set_roots(oz_engine* e, const uint64_t* black, const uint64_t* white, const int32_t* player);
/* num_sims x OthelloMCTS.simulate(root) for every game, strictly sequential per game (bit-exact mode).
 * OZ_PRIOR_HASH / OZ_PRIOR_NET run to completion; OZ_PRIOR_HOST returns after each wave of leaves:
 * *n_leaves > 0 means "evaluate them (oz_search_get_leaves / oz_search_put_priors) and call
 * oz_search_continue"; 0 means done.  OZ_ERR_NOMEM when a game's node pool / table filled up before its simulations
 * were done (the reference's dicts grow without bound, MCTS/__init__.py:19-28; here nodes_per_game bounds them). */
int oz_search_begin(oz_engine* e, int32_t num_sims, int32_t* n_leaves);
int oz_search_continue(oz_engine* e, int32_t* n_leaves);
/* Pending leaves in canonical form (the board passed to predict, othelo_mcts.py:82-88). HOST buffers. */
int oz_search_get_leaves(oz_engine* e, uint64_t* own, uint64_t* opp, int32_t n_leaves);
/* pi: [n_leaves][N*N] float32 probabilities in r*N+c order (Net/NNet.py:85-87), v: [n_leaves]. HOST buffers. */
int oz_search_put_priors(oz_engine* e, const float* pi, const float* v, int32_t n_leaves);
/* MCTS.N(state, action) for the root (MCTS/__init__.py:73-84): visits [n_games][64] by square bit, ns [n_games]. */
int oz_search_get_visits(oz_engine* e, int32_t* visits, int32_t* ns);
/* Root statistics of one game: q/p [64] doubles by square bit, qtag [64]: -1 not legal, 0 python int 0,
 * 1 python float, 2 numpy float32 (SURVEY A.4).  Returns OZ_ERR_STATE if the root is not in the tree. */
int oz_search_get_root_stats(oz_engine* e, int32_t game, double* q, double* p, int32_t* qtag);
int oz_search_get_status(oz_engine* e, int32_t* status);
/* counters: [0] simulations completed, [1] nodes expanded (= net evaluations, othelo_mcts.py:82-88),
 * [2] terminal visits, [3] evaluation-cache hits, [4] leaves that shared another game's evaluation, [5] max depth seen,
 * [6] transposition hits, [7] moves played. */
int oz_engine_counters(oz_engine* e, uint64_t* out8);

/* ---- search values (search and self-play) ------------------------------------------------- */
/* How a simulation backs a child's value up to the edge that led to it.  OZ_VALUES_REFERENCE (the default) negates it at
 * every ply, as the reference does: a move that finishes the game, or after which the opponent must pass, is credited
 * to the wrong side.  OZ_VALUES_STANDARD negates it only when the move swapped the side to move: a finished child is
 * worth +reward of the scoring to the edge that finished it, a child reached through a pass +v, every other child -v.
 * solve_leaves = K > 0 (OZ_VALUES_STANDARD and OZ_SCORING_STANDARD only): a new, non-finished child position below the
 * root with at most K empties is not expanded and not evaluated; its value is the sign (+1, 0, -1) of its perfect-play
 * margin for its side to move, backed up as an integer like a terminal and cached on the edge.  The root is never
 * solved.  Argument errors (unknown values, K outside [0, OZ_SOLVE_LEAVES_MAX], K > 0 without standard values and
 * standard scoring) fail with OZ_ERR_INVALID before any CUDA call.  Latched by the next oz_search_reset /
 * oz_selfplay_begin. */
#define OZ_VALUES_REFERENCE 0
#define OZ_VALUES_STANDARD 1
#define OZ_SOLVE_LEAVES_MAX 12
int oz_search_set_values(oz_engine* e, int32_t values, int32_t solve_leaves);
/* [0] leaves solved, [1] positions the leaf solver visited (each solved leaf, its children and their subtrees); cleared
 * with the other counters by oz_search_reset / oz_selfplay_begin. */
int oz_search_solve_counters(oz_engine* e, uint64_t* out2);

/* ---- root exploration (search and self-play) ------------------------------------------------ */
/* AlphaZero's two sources of exploration, both off by default.
 * Root noise (alpha > 0): a node gets Dirichlet(alpha) noise once, when it first serves as the root of a descent (the
 * root's second simulation when the first one created it, a self-play move onto a reused child, a root given by
 * oz_search_set_roots): its priors over its k legal moves become P'_j = (1 - fraction) * P_j + fraction * eta_j, in
 * double, each operation rounded separately, and a flag in the node header is set.  A flagged node is never noised
 * again (repeated oz_search_begin calls, oz_search_set_roots back to an old root); a noised node that later becomes an
 * interior node keeps its mixed priors.  k = 1 is only flagged.  The evaluation cache, the network outputs and the
 * other nodes are unchanged.
 * Noise stream, keyed by (seed, game id, root position) and independent of ply, slot, queue order, batch and cache:
 *   base = sm64(sm64(seed ^ 0x5EEDC01D) + game_id) (the self-play base below), rk = sm64(sm64(base ^ own) + opp) with
 *   (own, opp) the root's discs (side to move, other side; bit r*8+c); the j-th legal move (row-major) reads the words
 *   w_t = sm64(sm64(rk + j) + t), t = 0, 1, ..., in the order it uses uniforms u = ((w >> 11) + 1) * 2^-53 in (0, 1].
 *   g_j ~ Gamma(alpha): Marsaglia-Tsang on a = alpha + 1 if alpha < 1, else a = alpha: d = a - 1/3, c = 1 / sqrt(9d);
 *   repeat { z = polar normal (x = 2u - 1, y = 2u' - 1, s = xx + yy, retried unless 0 < s < 1, z = x sqrt(-2 log(s) / s));
 *   v = 1 + cz, retried if v <= 0; v = (vv)v; u; accept dv if u < 1 - (0.0331 z^2) z^2 or log u < 0.5 z^2 + d((1 - v) +
 *   log v) } (each loop gives up after 256 tries: the normal as 0, the gamma as d); alpha < 1: g = dv * exp(log(u) / alpha)
 *   with one more uniform.  eta_j = g_j / S, S = g_0 + g_1 + ... summed in ascending j (1/k if S = 0).
 *   log and exp are the engine's own, built from +, -, *, /, sqrt and integer operations (DESIGN.md 15).
 * Sampled moves (sample_moves = M, self-play only; no effect on the search API, which plays no moves): at move index
 * p < M the action is the first legal move (row-major) whose running visit sum exceeds
 * u = mulhi32(draw(p, 3) >> 32, sum of the root's visits); it replaces the first arg-max (temperature > 0) or the tie
 * draw (temperature == 0).  The e_greedy coin still applies on top.  The record's visit counts are unchanged.
 * NaN values, alpha outside [0, OZ_DIRICHLET_ALPHA_MAX], fraction outside [0, 1] or M outside [0, OZ_SAMPLE_MOVES_MAX]
 * fail with OZ_ERR_INVALID before any CUDA call.  (The bound on alpha keeps the sum S of up to 64 gamma variates, each
 * about alpha, far from overflow; a Dirichlet with alpha that large is the uniform distribution to double precision.)
 * Latched by the next oz_search_reset / oz_selfplay_begin. */
#define OZ_DIRICHLET_ALPHA_MAX 1e6
#define OZ_SAMPLE_MOVES_MAX 64
int oz_search_set_exploration(oz_engine* e, double alpha, double fraction, int32_t sample_moves);

/* ---- self-play: training.execute_episode (training.py:26-72) ------------------------------ */
/* Starts n_games episodes (start positions as oz_search_reset; a start whose side to move has no legal move is
 * rejected with OZ_ERR_INVALID).  temperature > 0: the greedy action is the first arg-max of the visit counts
 * (training.py:48-53).  temperature == 0 (the reference's setting from iteration `temperature_threshold` on,
 * main.py:73-76): the policy is one-hot on random.choice over the arg-max set (othelo_mcts.py:54-62) - a unique maximum
 * needs no draw, ties are drawn from the engine RNG.  With probability 1-e_greedy a uniformly random legal action is
 * played instead (training.py:55-56).  CPython's RNG stream is not reproduced; the engine's counter RNG is:
 *   base = sm64(sm64(seed ^ 0x5EEDC01D) + game_id); draw(p, w) = sm64(base + 4p + w) at move index p;
 *   tie-break tied[mulhi32(draw(p,2) >> 32, len(tied))] (row-major), coin (draw(p,0) >> 11) * 2^-53 <= e_greedy,
 *   random action legal[mulhi32(draw(p,1) >> 32, len(legal))].
 * tests/golden/episodes_rng.json holds the reference's own execute_episode run with these draws injected.
 * max_moves < 0: play to the end.
 * n_games may exceed max_games (a game QUEUE): the first max_games episodes start at once and a slot whose episode ends
 * takes the next queued game (fresh tree, its own RNG stream keyed by its game id, default id = game index), so the leaf
 * batch stays full over the whole job; start arrays then hold n_games entries.  Every game's result is independent of
 * the slot it ran in and of the other games (tests/test_gpu_search.py::test_game_queue_matches_separate_batches). */
int oz_selfplay_begin(oz_engine* e, int32_t n_games, const uint64_t* black, const uint64_t* white,
                      const int32_t* player, const uint64_t* game_ids, int32_t num_sims, double temperature,
                      double e_greedy, int32_t max_moves);
/* Runs `steps` engine steps (each: one tree kernel + one leaf-batch evaluation; every active game completes
 * >= 1 simulation per step).  steps < 0: run until every game has finished.  *n_active = games still running.
 * OZ_PRIOR_HOST is not supported here (use the search API). */
int oz_selfplay_run(oz_engine* e, int32_t steps, int32_t* n_active);
/* Per-move records of EVERY game of the job (queued ones included, indexed by game), HOST buffers sized [n_games][64]
 * (rec_visits [n_games][64][64], may be NULL unless log_visits): position before the move as black/white bitboards, action square bit, mover; n_moves,
 * winner (0 BLACK / 1 WHITE, draw -> BLACK, Othello/__init__.py:254-256; under OZ_SCORING_STANDARD a draw is
 * OZ_WINNER_DRAW (2); -1 unfinished) per game.
 * Entry n_moves[g] (< 64) of rec_black/rec_white[g] holds the position the episode ended in (the board every example
 * of the reference aliases, training.py:63). */
int oz_selfplay_get_records(oz_engine* e, uint64_t* rec_black, uint64_t* rec_white, uint8_t* rec_action,
                            uint8_t* rec_player, int32_t* n_moves, int32_t* winner, int32_t* rec_visits);
/* Current positions of the min(n_games, max_games) slots (HOST buffers; any may be NULL). */
int oz_selfplay_get_positions(oz_engine* e, uint64_t* black, uint64_t* white, int32_t* player);

/* ---- network: NNetWrapper.predict / OthelloNN (Net/NNet.py:70-87, Net/OthelloNN.py:42-52) -- */
/* Weights as one float32 HOST blob in Keras layer order (kernel HWIO / (in,out), bias, then BN gamma, beta,
 * moving_mean, moving_var for the six BN layers): see INTEGRATION.md for the exact order.  BN (eps 1e-3) is
 * folded, conv2..fc2 + heads are cast to bf16, and the conv1 / conv1∘conv2 lookup tables are rebuilt on the device
 * (19683 x 9 x channels bf16, ~0.1 ms).  channels must be a multiple of 128. */
int oz_net_load_weights(oz_engine* e, const float* blob, int64_t n_floats, int32_t channels);
/* Same, from a DEVICE float32 blob (e.g. a tensor just received by ncclBroadcast). */
int oz_net_load_weights_dev(oz_engine* e, const float* blob_dev, int64_t n_floats, int32_t channels);
int64_t oz_net_blob_floats(int32_t board_size, int32_t channels);
/* FP8 evaluation (DESIGN.md 13): OR OZ_NET_FP8 into the `channels` argument of oz_net_load_weights[_dev] and
 * oz_dist_broadcast_weights to run conv3, conv4 and fc1 on e4m3 operands (per-output-channel weight scales, one static
 * scale per input activation calibrated at load, fp32 accumulation).  Everything else stays bf16 and the blob format is
 * unchanged (oz_net_blob_floats takes the plain channel count).  FP8 needs channels to be a multiple of 256 and the
 * default kernels: with OZ_NET_CONV2=gemm, OZ_NET_CONV3=wino or OZ_NET_NO_2SM=1 in the environment an FP8 load fails
 * with OZ_ERR_STATE.  The precision is fixed by an engine's first load, like the channel count: a later load with the
 * other precision fails with OZ_ERR_STATE. */
#define OZ_NET_FP8 0x10000
/* Scales of the loaded FP8 network into a HOST buffer of 3 + 2 * channels + 1024 floats: sa_2, sa_3, sa_4 (the static
 * scales of act2, act3, act4 = the inputs of conv3, conv4, fc1), then the per-output-channel weight scales of conv3
 * [channels], conv4 [channels] and fc1 [1024].  A real value x is stored as e4m3_rn(x / scale).  OZ_ERR_STATE unless the
 * engine's weights were loaded with OZ_NET_FP8. */
int oz_net_fp8_scales(oz_engine* e, float* out);
/* Batched predict on canonical boards. pi: [n][N*N] softmax probabilities (r*N+c), logits same shape (may be
 * NULL), v: [n] tanh.  HOST buffers (rows of N*N floats) / DEVICE buffers (rows padded to a stride of 64 floats). */
int oz_net_forward_host(oz_engine* e, const uint64_t* own, const uint64_t* opp, int32_t n, float* pi,
                        float* logits, float* v);
int oz_net_forward_dev(oz_engine* e, const uint64_t* own, const uint64_t* opp, int32_t n, float* pi,
                       float* logits, float* v);
/* Debug/inspection: raw bf16 activations of the last forward. layer 0..5 = conv1, conv2, conv3, conv4, fc1, fc2
 * outputs ([n][rows][channels] row-major); copies `bytes` bytes to the HOST buffer.  An FP8 network (OZ_NET_FP8) stores
 * layers 1..3 (act2, act3, act4) as raw e4m3 bytes, one per element, in units of their scales (oz_net_fp8_scales); layers
 * 4 and 5 stay bf16.  conv1+conv2 normally run as one
 * gather over a pre-computed partial-product table (DESIGN.md 3a), which never materialises conv1's output: layer 0 then
 * fails with OZ_ERR_STATE (engines created with OZ_NET_CONV2=gemm in the environment keep it); likewise layer 1 with the
 * opt-in OZ_NET_CONV3=wino (conv3 as a Winograd F(2,3) kernel fed by the gather's input transform, DESIGN.md 3b). */
int oz_net_get_activation(oz_engine* e, int32_t layer, void* host_bf16, int64_t bytes);
/* Kernel launches issued by this engine since creation (bench.py "gpu_launches"). */
int oz_engine_launches(oz_engine* e, uint64_t* launches);
/* Per-layer device timing with CUDA events on the engine stream (no host sync in the hot loop).
 * oz_net_layer_times: average ms per launch since the previous call for [0] conv1 gather (0 when conv1+conv2 run as
 * the table gather), [1] conv2 (the table gather, or the implicit GEMM), [2] conv3, [3] conv4, [4] fc1, [5] fc2,
 * [6] heads; [7] = number of forwards averaged. */
int oz_net_set_timing(oz_engine* e, int32_t on);
int oz_net_layer_times(oz_engine* e, float* ms8);

/* ---- dist: the two collectives of an iteration, over NCCL (one process per GPU) ---------------------- */
/* C1 replaces the reference's weight fan-out (workers.py:203-296: temp .h5 -> sftp -> scp tree), C2 its result gather
 * (pickled stdout, workers.py:147-159,180-184).  Nothing is exchanged while games are played (they shard by id).
 * NCCL is resolved at run time (dlopen libnccl.so.2); without it these calls fail with OZ_ERR_STATE.
 * oz_dist_unique_id: rank 0 creates the 128-byte ncclUniqueId, the host ships it to the other ranks (any channel);
 * oz_dist_init: every rank joins (collective; the communicator lives on the engine's device and stream). */
int oz_dist_unique_id(uint8_t* id128);
int oz_dist_init(oz_engine* e, int32_t rank, int32_t world, const uint8_t* id128);
int oz_dist_destroy(oz_engine* e);
/* C1 (collective): `root` passes the float32 HOST blob (oz_net_load_weights' format), the others may pass NULL; every rank
 * ends with the weights folded and loaded on its device (and its evaluation cache cleared). */
int oz_dist_broadcast_weights(oz_engine* e, const float* blob, int64_t n_floats, int32_t channels, int32_t root);
/* C2 (collective): every rank contributes n_rows packed example rows (3 x uint64 per position: black, white,
 * action | player<<8 | winner<<16 | game<<32 - othellozero_b200.dist.pack_records) from a HOST buffer and receives the
 * concatenation in rank order in out_rows (HOST, capacity_rows rows); *total_rows = rows gathered.  out_rows = NULL only
 * queries the total (still collective). */
int oz_dist_gather_examples(oz_engine* e, const uint64_t* rows, int64_t n_rows, uint64_t* out_rows, int64_t capacity_rows,
                            int64_t* total_rows);

/* ---- measurement aid (bench.py) ---------------------------------------------------------------------- */
/* L2 read bandwidth of `device`, GB/s: `passes` sweeps of 16-byte loads over an L2-resident buffer of `megabytes` MB
 * (B200: 126 MB of L2), timed with CUDA events.  The denominator of the conv1∘conv2 table gather's roofline: that kernel
 * is bound by the L2 -> SM path, not by HBM.  (No reference counterpart: the reference has no kernels to measure.) */
int oz_probe_l2_read(int32_t device, int32_t megabytes, int32_t passes, double* gb_per_s);

#ifdef __cplusplus
}
#endif
#endif /* OZ_B200_H */
