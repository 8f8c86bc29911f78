// oz_engine.cuh — internal engine state shared by the tree, net and C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/oz_b200.h"
#include "oz_bitboard.cuh"

typedef unsigned long long u64;
typedef unsigned int u32;

// ---- error plumbing ------------------------------------------------------------------------
void oz_set_error(const char* fmt, ...);
#define OZ_CUDA(expr)                                                                              \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            oz_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return OZ_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)
#define OZ_REQUIRE(cond, ...)        \
    do {                             \
        if (!(cond)) {               \
            oz_set_error(__VA_ARGS__); \
            return OZ_ERR_INVALID;   \
        }                            \
    } while (0)

// ---- host-buffer entry points: per-thread device scratch + pinned staging + stream (oz_rules.cu, oz_solve.cu) ----------
struct OzHostScratch {
    int device = -1;
    unsigned char* dev = nullptr;
    unsigned char* pin = nullptr;
    size_t cap = 0;
    cudaStream_t st = nullptr;
    void release() {
        if (dev) cudaFree(dev);
        if (pin) cudaFreeHost(pin);
        if (st) cudaStreamDestroy(st);
        dev = pin = nullptr; st = nullptr; cap = 0; device = -1;
    }
    ~OzHostScratch() { release(); }  // at thread exit; errors after runtime teardown are ignored
    int reserve(int dev_id, size_t bytes) {
        cudaError_t e = cudaSetDevice(dev_id);
        if (e != cudaSuccess) { oz_set_error("cudaSetDevice(%d) failed: %s", dev_id, cudaGetErrorString(e)); return OZ_ERR_CUDA; }
        if (device != dev_id) release();
        if (!st) {
            e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
            if (e != cudaSuccess) { oz_set_error("cudaStreamCreate failed: %s", cudaGetErrorString(e)); return OZ_ERR_CUDA; }
            device = dev_id;
        }
        if (bytes <= cap) return OZ_OK;
        size_t want = cap ? cap : 4096;
        while (want < bytes) want *= 2;
        if (dev) cudaFree(dev);
        if (pin) cudaFreeHost(pin);
        dev = pin = nullptr; cap = 0;
        e = cudaMalloc((void**)&dev, want);
        if (e == cudaSuccess) e = cudaMallocHost((void**)&pin, want);
        if (e != cudaSuccess) {
            oz_set_error("scratch allocation of %zu bytes failed: %s", want, cudaGetErrorString(e));
            if (dev) cudaFree(dev);
            dev = nullptr;
            return OZ_ERR_NOMEM;
        }
        cap = want;
        return OZ_OK;
    }
};
inline size_t oz_up256(size_t x) { return (x + 255) & ~(size_t)255; }
OzHostScratch& oz_host_scratch();

// Scorings of the tree kernel (instantiated per scoring, chosen at launch): REFERENCE counts a draw as a BLACK win,
// STANDARD scores it as a draw (value 0, winner code OZ_WINNER_DRAW).
enum : int { SCORING_REFERENCE = 0, SCORING_STANDARD = 1 };
// Value conventions of the tree kernel (instantiated per convention, chosen at launch; oz_search_set_values).
enum : int { VALUES_REFERENCE = OZ_VALUES_REFERENCE, VALUES_STANDARD = OZ_VALUES_STANDARD };

// The board_size argument of the C-ABI: N (4, 6 or 8), optionally | OZ_RULES_STANDARD | OZ_SCORING_STANDARD.  -> N, the
// ozbb rule set and the scoring (any output may be null); any other bit is OZ_ERR_INVALID.  Only the C-ABI entry points
// see the flags.
inline int oz_decode_board(int32_t board_size, int* n, int* rules, int* scoring = nullptr) {
    const int size = board_size & ~(OZ_RULES_STANDARD | OZ_SCORING_STANDARD);
    if (size != 4 && size != 6 && size != 8) {
        oz_set_error("board_size must be 4, 6 or 8, optionally | OZ_RULES_STANDARD | OZ_SCORING_STANDARD (got %d)",
                     board_size);
        return OZ_ERR_INVALID;
    }
    if (n) *n = size;
    if (rules) *rules = (board_size & OZ_RULES_STANDARD) ? ozbb::RULES_STANDARD : ozbb::RULES_REFERENCE;
    if (scoring) *scoring = (board_size & OZ_SCORING_STANDARD) ? SCORING_STANDARD : SCORING_REFERENCE;
    return OZ_OK;
}

// ---- tree node pool layout (HBM) -----------------------------------------------------------------
// Node = 48-byte header followed by SoA child rows, k = popcount(legal):
//   double P[k]; double Q[k]; int N[k]; int child[k];        (48 + 24k bytes, rounded up to 16)
// Child slot j <-> j-th set bit of `legal` (ascending == reference row-major action order).
// Node references are offsets into the game's arena in 16-byte units.
struct __align__(16) OzNodeHdr {
    u64 own, opp;  // canonical key (exact board; MCTS/__init__.py:7-16 hashes the board bytes)
    u64 legal;     // cached get_state_actions (MCTS/__init__.py:183-187)
    u64 qf32;      // bit j: Q[j] currently has numpy float32 type (else python float / int 0)
    int ns;        // _Ns
    int k;
    int vns;       // in-flight (virtual) visits through this node; 0 outside a virtual-loss wave
    int pad1;      // 1: the node has served as a root with exploration on (its noise is mixed in); 0 otherwise
};
static_assert(sizeof(OzNodeHdr) == 48, "node header layout");

constexpr int OZ_CH_UNKNOWN = -1;   // edge never traversed
constexpr int OZ_CH_TERM_NEG = -2;  // child is terminal, simulate() returns -1
constexpr int OZ_CH_TERM_POS = -3;  // child is terminal, simulate() returns +1
constexpr int OZ_CH_PENDING = -4;   // leaf emitted by the current virtual-loss wave, not expanded yet
constexpr int OZ_CH_TERM_DRAW = -5; // child is a drawn terminal, simulate() returns 0 (standard scoring only)
constexpr int OZ_MAX_DEPTH = 64;

struct OzTreeParams {
    int n;          // board size
    int nsq;        // n*n
    u64 full;       // full_mask(n)
    int G;          // active game slots
    int prior_mode;
    int selfplay;   // 1: move transitions happen on device
    int log_visits;
    double c;
    // per-slot state
    u64* black; u64* white; int* player;
    int* status; int* root_node; int* sims_left; int* ply; u64* game_id; int* winner;
    // pending leaf (WAIT_LEAF)
    u64* pend_own; u64* pend_opp; u64* pend_legal;
    int* pend_parent; int* pend_edge; int* pend_depth; int* pend_leaf;  // [G][vl_width]
    int* pend_count;                                                     // [G] leaves of the current wave
    int vl_width;                                                        // 1 = sequential (bit-exact) mode
    int sim_budget;  // self-play with an evaluator: simulations a game may complete per launch WITHOUT needing the evaluator
                     // (terminal visits, evaluation-cache hits) before it yields to the next step; 0 = unbounded
    long long time_budget;  // ... and the age of the launch (SM clocks) after which such a game yields; 0 = unbounded
    u32* path_node; u32* path_edge;  // [G][vl_width][64]
    // pools
    unsigned char* arena; u64 arena_stride;  // bytes per game
    u32* bump;                                // next free offset (16-byte units) per game
    u64* table; int table_log2;               // [G][1<<table_log2] : fingerprint<<32 | (node_off+1)
    // leaf batch
    u64* leaf_own; u64* leaf_opp; int* leaf_count; const float* leaf_pi; const float* leaf_v;
    int* leaf_count_next;  // self-play: the counter of the next step, cleared by this step's tree kernel (or null)
    // cross-game evaluation cache (optional)
    u64* cache_tags; u64* cache_keys; int* cache_leaf; float* cache_pi; float* cache_v; int* leaf_cache_idx;
    int cache_log2_buckets;
    // self-play
    int num_sims; int max_moves; double e_greedy; double temperature; u64 seed;
    u64* rec_black; u64* rec_white; unsigned char* rec_action; unsigned char* rec_player; int* rec_visits;
    int* rec_nmoves;  // [record capacity] plies played so far, by game index
    // game queue: a slot whose episode ends starts game *next_game (while < total_games) - self-play keeps the leaf batch
    // full over a job of more games than slots.  Records / winner / rec_nmoves are indexed by GAME (slot_game[slot]).
    int total_games;
    int* next_game;
    int* slot_game;                                          // [G]
    const u64* q_black; const u64* q_white; const int* q_player; const u64* q_ids;  // [total_games] start positions or null
    // counters (device)
    u64* counters;  // see oz_engine_counters
    int* n_active;
    // standard values only (appended: the fields above keep their offsets in the kernel's parameter block)
    int solve_leaves;            // K: new child positions below the root with <= K empties are solved, not expanded
    u64 corners, near_corners;   // the leaf solver's move ordering (oz_ordering_masks)
    u64* solve_counters;         // [0] leaves solved, [1] solver positions (oz_search_solve_counters)
    // root exploration only (appended likewise; oz_search_set_exploration)
    double dir_alpha, dir_fraction;  // Dirichlet noise mixed into each root's priors once; alpha = 0: none
    int sample_moves;                // self-play plies p < M play a move drawn in proportion to the root visit counts
};

struct OzNet;  // oz_net.cu

struct oz_engine {
    oz_engine_config cfg;      // cfg.board_size holds plain N; the flags of the caller's value are in `rules`, `scoring`
    int rules = ozbb::RULES_REFERENCE;
    int scoring = SCORING_REFERENCE;
    int values = VALUES_REFERENCE;    // latched from the requested values by oz_tree_reset(clear)
    int values_req = VALUES_REFERENCE, solve_leaves_req = 0;  // oz_search_set_values
    double dir_alpha_req = 0.0, dir_fraction_req = 0.0;       // oz_search_set_exploration, latched like the values
    int sample_moves_req = 0;
    cudaStream_t stream = nullptr;
    OzTreeParams tp{};
    int n_games = 0;
    bool search_started = false;
    int host_leaves = 0;
    int table_log2 = 0;
    u64 arena_stride = 0;
    u64 launches = 0;
    size_t cache_entries = 0;
    int max_leaves = 0;        // max_games * vl_width: capacity of the leaf batch and of the network
    int rec_games = 0;         // games whose records the last oz_selfplay_begin covers (>= n_games slots with a queue)
    size_t rec_capacity = 0;   // games the record buffers hold (grown on demand, see oz_tree_reserve_records)
    void* rec_buf = nullptr;   // one allocation behind tp.rec_* / tp.winner / tp.rec_nmoves
    void* q_buf = nullptr;     // queued start positions of the current self-play job (grow-only)
    size_t q_bytes = 0;
    unsigned char* scratch = nullptr;  // persistent device staging for the host-buffer entry points (no per-call
    size_t scratch_bytes = 0;          // cudaMallocAsync/FreeAsync: measured 2-350 ms per call when the pool is trimmed)
    // device allocations (freed in destroy)
    void* allocs[64];
    int n_allocs = 0;
    float* leaf_pi = nullptr;  // [max_games][64]
    float* leaf_v = nullptr;
    float* leaf_logits = nullptr;
    int* h_pinned = nullptr;   // small pinned scratch
    int* leaf_count_base = nullptr;  // [8]: [0] leaf count, [1] net-forward count, [2] waiting games, [3] bad start, [4] second leaf count (self-play ping-pong)
    OzNet* net = nullptr;
    float layer_ms[8] = {0};
    void* comm = nullptr;      // ncclComm_t of oz_dist_init (oz_dist.cu), or null
    int dist_rank = 0, dist_world = 1;
};

// tree (oz_tree.cu)
int oz_tree_alloc(oz_engine* e);
int oz_tree_reset(oz_engine* e, int n_games, const u64* black, const u64* white, const int* player, const u64* ids,
                  bool clear);
int oz_tree_step(oz_engine* e);  // one tree kernel launch
int oz_tree_reserve_records(oz_engine* e, size_t games);
int oz_tree_visits(oz_engine* e, int* visits_dev, int* ns_dev);
int oz_tree_root_stats(oz_engine* e, int game, double* q_dev, double* p_dev, int* tag_dev);
int oz_tree_hash_eval(oz_engine* e);      // wave mode + closed-form priors: evaluate the parked leaves
int oz_tree_cache_clear(oz_engine* e);    // weights changed

// net (oz_net.cu)
int oz_net_create(oz_engine* e);
void oz_net_destroy(oz_engine* e);
int oz_net_load(oz_engine* e, const float* blob, int64_t n_floats, int channels, bool on_device);
// forward over `count_dev` (device int, <= max_games) canonical boards -> e->leaf_pi / leaf_logits / leaf_v
// publish = true: the heads epilogue also copies every cache OWNER's priors into its evaluation-cache entry and marks
// it ready (what cache_publish_kernel did in a launch of its own)
int oz_net_forward(oz_engine* e, const u64* own_dev, const u64* opp_dev, const int* count_dev, int max_count,
                   float* pi_dev, float* logits_dev, float* v_dev, bool publish = false);
int64_t oz_net_blob_floats_impl(int board_size, int channels);
int oz_net_activation(oz_engine* e, int layer, void* host, int64_t bytes);
int oz_net_scales(oz_engine* e, float* out);
void oz_net_set_timing_impl(oz_engine* e, bool on);
int oz_net_times(oz_engine* e, float* ms8);

template <typename T>
int oz_dev_alloc(oz_engine* e, T** p, size_t count) {
    void* q = nullptr;
    cudaError_t err = cudaMalloc(&q, count * sizeof(T) + 16);
    if (err != cudaSuccess) {
        oz_set_error("cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(err));
        return OZ_ERR_NOMEM;
    }
    if (e->n_allocs >= 64) { oz_set_error("too many allocations"); return OZ_ERR_NOMEM; }
    e->allocs[e->n_allocs++] = q;
    *p = (T*)q;
    return OZ_OK;
}
