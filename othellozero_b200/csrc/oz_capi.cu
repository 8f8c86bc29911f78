// oz_capi.cu — the C-ABI (include/oz_b200.h): engine lifetime, search / self-play drivers, net entry points.
#include <stdarg.h>
#include <string.h>

#include "oz_engine.cuh"

static thread_local char g_err[512] = "";

void oz_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* oz_last_error(void) { return g_err; }
extern "C" int oz_abi_version(void) { return OZ_ABI_VERSION; }

extern "C" int oz_device_count(int32_t* count) {
    OZ_REQUIRE(count != nullptr, "count is NULL");
    int c = 0;
    cudaError_t err = cudaGetDeviceCount(&c);
    if (err != cudaSuccess) {
        *count = 0;
        oz_set_error("cudaGetDeviceCount failed: %s (this library has no CPU fallback)", cudaGetErrorString(err));
        return OZ_ERR_CUDA;
    }
    *count = c;
    return OZ_OK;
}

// ---- small device helpers ---------------------------------------------------------------------------
__global__ void search_begin_kernel(OzTreeParams P, int num_sims) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= P.G) return;
    int st = P.status[g];
    if (st == OZ_GAME_IDLE || st == OZ_GAME_ACTIVE) {
        P.status[g] = OZ_GAME_ACTIVE;
        P.sims_left[g] = num_sims;
    }
}

__global__ void scatter_priors_kernel(float* __restrict__ dst, const float* __restrict__ src, int n_leaves, int nsq) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_leaves * nsq) return;
    int l = i / nsq, f = i - l * nsq;
    dst[(size_t)l * 64 + f] = src[i];
}

// Start positions of a self-play job: *bad = lowest index of a position that cannot be played.
__global__ void validate_starts_kernel(int n_games, const u64* __restrict__ black, const u64* __restrict__ white,
                                       const int* __restrict__ player, u64 full, int* bad) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_games) return;
    const u64 b = black[g], w = white[g];
    const int pl = player ? player[g] : 0;
    const bool ok = !(b & w) && !((b | w) & ~full) && (pl == 0 || pl == 1) &&
                    ozbb::legal_moves(pl ? w : b, pl ? b : w, full) != 0ull;
    if (!ok) atomicMin(bad, g);
}

// ---- engine -----------------------------------------------------------------------------------------
extern "C" int oz_engine_create(const oz_engine_config* cfg, oz_engine** out) {
    OZ_REQUIRE(cfg && out, "null argument");
    *out = nullptr;
    int size, rules, scoring;
    if (oz_decode_board(cfg->board_size, &size, &rules, &scoring)) return OZ_ERR_INVALID;
    OZ_REQUIRE(cfg->max_games >= 1 && cfg->max_games <= (1 << 20), "max_games out of range: %d", cfg->max_games);
    OZ_REQUIRE(cfg->nodes_per_game >= 2 && cfg->nodes_per_game <= (1 << 22), "nodes_per_game out of range: %d",
               cfg->nodes_per_game);
    OZ_REQUIRE(cfg->prior_mode >= OZ_PRIOR_HASH && cfg->prior_mode <= OZ_PRIOR_NET, "bad prior_mode %d", cfg->prior_mode);
    OZ_REQUIRE(cfg->prior_mode != OZ_PRIOR_NET || size >= 6, "the network needs board_size 6 or 8");
    OZ_REQUIRE(cfg->vl_width >= 0 && cfg->vl_width <= 64, "vl_width out of range: %d", cfg->vl_width);
    int ndev = 0;
    int rc = oz_device_count(&ndev);
    if (rc) return rc;
    if (cfg->device < 0 || cfg->device >= ndev) {
        oz_set_error("device %d not available (%d CUDA devices; no CPU fallback)", cfg->device, ndev);
        return OZ_ERR_CUDA;
    }
    OZ_CUDA(cudaSetDevice(cfg->device));
    oz_engine* e = new oz_engine();
    e->cfg = *cfg;
    e->cfg.board_size = size;
    e->rules = rules;
    e->scoring = scoring;
    cudaError_t err = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
    if (err != cudaSuccess) {
        oz_set_error("cudaStreamCreate failed: %s", cudaGetErrorString(err));
        delete e;
        return OZ_ERR_CUDA;
    }
    rc = oz_tree_alloc(e);
    if (!rc) {
        err = cudaMallocHost((void**)&e->h_pinned, 64 * sizeof(int));
        if (err != cudaSuccess) { oz_set_error("cudaMallocHost failed: %s", cudaGetErrorString(err)); rc = OZ_ERR_CUDA; }
    }
    if (!rc) rc = oz_net_create(e);
    if (rc) {
        oz_engine_destroy(e);
        return rc;
    }
    err = cudaStreamSynchronize(e->stream);
    if (err != cudaSuccess) {
        oz_set_error("engine init failed: %s", cudaGetErrorString(err));
        oz_engine_destroy(e);
        return OZ_ERR_CUDA;
    }
    *out = e;
    return OZ_OK;
}

extern "C" int oz_engine_destroy(oz_engine* e) {
    if (!e) return OZ_OK;
    cudaSetDevice(e->cfg.device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    oz_dist_destroy(e);
    oz_net_destroy(e);
    for (int i = 0; i < e->n_allocs; ++i) cudaFree(e->allocs[i]);
    if (e->rec_buf) cudaFree(e->rec_buf);
    if (e->q_buf) cudaFree(e->q_buf);
    if (e->h_pinned) cudaFreeHost(e->h_pinned);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
    return OZ_OK;
}

extern "C" int oz_engine_sync(oz_engine* e) {
    OZ_REQUIRE(e, "null engine");
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

extern "C" void* oz_engine_stream(oz_engine* e) { return e ? (void*)e->stream : nullptr; }

extern "C" int oz_engine_counters(oz_engine* e, uint64_t* out8) {
    OZ_REQUIRE(e && out8, "null argument");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    OZ_CUDA(cudaMemcpyAsync(out8, e->tp.counters, 8 * sizeof(u64), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

extern "C" int oz_search_set_values(oz_engine* e, int32_t values, int32_t solve_leaves) {
    OZ_REQUIRE(e, "null engine");
    OZ_REQUIRE(values == OZ_VALUES_REFERENCE || values == OZ_VALUES_STANDARD,
               "values must be OZ_VALUES_REFERENCE or OZ_VALUES_STANDARD (got %d)", values);
    OZ_REQUIRE(solve_leaves >= 0 && solve_leaves <= OZ_SOLVE_LEAVES_MAX, "solve_leaves must be in [0, %d] (got %d)",
               OZ_SOLVE_LEAVES_MAX, solve_leaves);
    // under reference scoring a drawn final position is worth +1 to whoever moved last: not a function of the margin
    OZ_REQUIRE(solve_leaves == 0 || (values == OZ_VALUES_STANDARD && e->scoring == SCORING_STANDARD),
               "solve_leaves > 0 needs standard values and standard scoring (OZ_SCORING_STANDARD)");
    e->values_req = values;
    e->solve_leaves_req = solve_leaves;
    return OZ_OK;
}

extern "C" int oz_search_set_exploration(oz_engine* e, double alpha, double fraction, int32_t sample_moves) {
    OZ_REQUIRE(e, "null engine");
    OZ_REQUIRE(alpha >= 0.0 && alpha <= OZ_DIRICHLET_ALPHA_MAX, "dirichlet alpha must be in [0, %g] (got %g)",
               OZ_DIRICHLET_ALPHA_MAX, alpha);
    OZ_REQUIRE(fraction >= 0.0 && fraction <= 1.0, "dirichlet fraction must be in [0, 1] (got %g)", fraction);
    OZ_REQUIRE(sample_moves >= 0 && sample_moves <= OZ_SAMPLE_MOVES_MAX, "sample_moves must be in [0, %d] (got %d)",
               OZ_SAMPLE_MOVES_MAX, sample_moves);
    e->dir_alpha_req = alpha;
    e->dir_fraction_req = fraction;
    e->sample_moves_req = sample_moves;
    return OZ_OK;
}

extern "C" int oz_search_solve_counters(oz_engine* e, uint64_t* out2) {
    OZ_REQUIRE(e && out2, "null argument");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    OZ_CUDA(cudaMemcpyAsync(out2, e->tp.solve_counters, 2 * sizeof(u64), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

extern "C" int oz_engine_launches(oz_engine* e, uint64_t* launches) {
    OZ_REQUIRE(e && launches, "null argument");
    *launches = e->launches;
    return OZ_OK;
}

// ---- search -----------------------------------------------------------------------------------------
extern "C" int oz_search_reset(oz_engine* e, int32_t n_games, const uint64_t* black, const uint64_t* white,
                               const int32_t* player, const uint64_t* game_ids) {
    OZ_REQUIRE(e, "null engine");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    e->tp.selfplay = 0;
    e->tp.leaf_count = e->leaf_count_base;
    e->tp.leaf_count_next = nullptr;
    e->search_started = false;
    int rc = oz_tree_reset(e, n_games, (const u64*)black, (const u64*)white, player, (const u64*)game_ids, true);
    if (rc) return rc;
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

extern "C" int oz_search_set_roots(oz_engine* e, const uint64_t* black, const uint64_t* white, const int32_t* player) {
    OZ_REQUIRE(e && black && white, "null argument");
    OZ_REQUIRE(e->n_games > 0, "oz_search_reset first");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    int rc = oz_tree_reset(e, e->n_games, (const u64*)black, (const u64*)white, player, nullptr, false);
    if (rc) return rc;
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

static int read_leaf_count(oz_engine* e, int* n) {
    OZ_CUDA(cudaMemcpyAsync(e->h_pinned, e->tp.leaf_count, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    *n = e->h_pinned[0];
    return OZ_OK;
}

__global__ void count_status_kernel(const OzTreeParams P, int wanted, int* out) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < P.G && P.status[g] == wanted) atomicAdd(out, 1);
}

static int count_status(oz_engine* e, int wanted, int* n) {
    int* d = e->leaf_count_base + 2;
    OZ_CUDA(cudaMemsetAsync(d, 0, sizeof(int), e->stream));
    count_status_kernel<<<(e->tp.G + 255) / 256, 256, 0, e->stream>>>(e->tp, wanted, d);
    OZ_CUDA(cudaGetLastError());
    e->launches++;
    OZ_CUDA(cudaMemcpyAsync(&e->h_pinned[4], d, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    *n = e->h_pinned[4];
    return OZ_OK;
}

// Evaluate the pending leaf batch with the device network (count stays on the device).
static int eval_leaves_net(oz_engine* e) {
    // the heads kernel's epilogue publishes the new evaluation-cache entries (no separate cache_publish launch)
    // (no logits: the search consumes probabilities and the value only)
    return oz_net_forward(e, e->tp.leaf_own, e->tp.leaf_opp, e->tp.leaf_count, e->n_games * e->tp.vl_width, e->leaf_pi, nullptr,
                          e->leaf_v, e->tp.cache_tags != nullptr);
}

// Evaluate the parked leaves with whatever this engine's prior source is (device network / closed-form hash).
static int eval_leaves(oz_engine* e) {
    if (e->cfg.prior_mode == OZ_PRIOR_NET) return eval_leaves_net(e);
    return oz_tree_hash_eval(e);
}

static int search_pump(oz_engine* e, int32_t* n_leaves) {
    OzTreeParams& P = e->tp;
    const int mode = e->cfg.prior_mode;
    const bool inline_hash = mode == OZ_PRIOR_HASH && P.vl_width <= 1;  // whole search inside one launch
    while (true) {
        OZ_CUDA(cudaMemsetAsync(P.leaf_count, 0, sizeof(int), e->stream));
        int rc = oz_tree_step(e);
        if (rc) return rc;
        if (inline_hash) { *n_leaves = 0; break; }
        // finished when no game is parked any more (a wave made only of cache hits parks games without emitting leaves)
        int nl = 0;
        if ((rc = read_leaf_count(e, &nl))) return rc;
        if (mode == OZ_PRIOR_HOST) {
            if (nl == 0) { *n_leaves = 0; break; }
            e->host_leaves = nl; *n_leaves = nl; return OZ_OK;
        }
        int waiting = 0;
        if ((rc = count_status(e, OZ_GAME_WAIT_LEAF, &waiting))) return rc;
        if (waiting == 0) { *n_leaves = 0; break; }
        if (nl > 0 && (rc = eval_leaves(e))) return rc;
    }
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    e->host_leaves = 0;
    // a game whose node pool or table filled up stopped short of num_sims: report it instead of returning thinner counts
    int full = 0;
    int rc = count_status(e, OZ_GAME_POOL_FULL, &full);
    if (rc) return rc;
    if (full > 0) {
        oz_set_error("node pool exhausted in %d game(s) before the requested simulations were done (nodes_per_game = %d "
                     "is sized for 16 children per node on average)", full, e->cfg.nodes_per_game);
        return OZ_ERR_NOMEM;
    }
    return OZ_OK;
}

extern "C" int oz_search_begin(oz_engine* e, int32_t num_sims, int32_t* n_leaves) {
    OZ_REQUIRE(e && n_leaves, "null argument");
    OZ_REQUIRE(num_sims >= 1, "num_sims must be >= 1");
    if (e->n_games <= 0) { oz_set_error("oz_search_reset first"); return OZ_ERR_STATE; }
    if (e->host_leaves) { oz_set_error("pending leaves have not been answered"); return OZ_ERR_STATE; }
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    e->tp.selfplay = 0;
    e->tp.leaf_count = e->leaf_count_base;
    e->tp.leaf_count_next = nullptr;
    search_begin_kernel<<<(e->tp.G + 255) / 256, 256, 0, e->stream>>>(e->tp, num_sims);
    OZ_CUDA(cudaGetLastError());
    e->launches++;
    return search_pump(e, n_leaves);
}

extern "C" int oz_search_continue(oz_engine* e, int32_t* n_leaves) {
    OZ_REQUIRE(e && n_leaves, "null argument");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    if (e->host_leaves) { oz_set_error("pending leaves have not been answered (oz_search_put_priors)"); return OZ_ERR_STATE; }
    return search_pump(e, n_leaves);
}

extern "C" int oz_search_get_leaves(oz_engine* e, uint64_t* own, uint64_t* opp, int32_t n_leaves) {
    OZ_REQUIRE(e && own && opp, "null argument");
    OZ_REQUIRE(n_leaves >= 0 && n_leaves <= e->host_leaves, "n_leaves %d > pending %d", n_leaves, e->host_leaves);
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    OZ_CUDA(cudaMemcpyAsync(own, e->tp.leaf_own, (size_t)n_leaves * 8, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(opp, e->tp.leaf_opp, (size_t)n_leaves * 8, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

extern "C" int oz_search_put_priors(oz_engine* e, const float* pi, const float* v, int32_t n_leaves) {
    OZ_REQUIRE(e && pi && v, "null argument");
    if (n_leaves != e->host_leaves) {
        oz_set_error("expected priors for %d leaves, got %d", e->host_leaves, n_leaves);
        return OZ_ERR_STATE;
    }
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    const int nsq = e->tp.nsq;
    float* tmp = (float*)e->scratch;  // n_leaves <= max_leaves rows of nsq <= 64 floats
    OZ_CUDA(cudaMemcpyAsync(tmp, pi, (size_t)n_leaves * nsq * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    scatter_priors_kernel<<<(n_leaves * nsq + 255) / 256, 256, 0, e->stream>>>(e->leaf_pi, tmp, n_leaves, nsq);
    OZ_CUDA(cudaGetLastError());
    e->launches++;
    OZ_CUDA(cudaMemcpyAsync(e->leaf_v, v, (size_t)n_leaves * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    e->host_leaves = 0;
    return OZ_OK;
}

extern "C" int oz_search_get_visits(oz_engine* e, int32_t* visits, int32_t* ns) {
    OZ_REQUIRE(e && visits && ns, "null argument");
    OZ_REQUIRE(e->n_games > 0, "oz_search_reset first");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    size_t nv = (size_t)e->n_games * 64;
    int* dv = (int*)e->scratch;
    int rc = oz_tree_visits(e, dv, dv + nv);
    if (rc) return rc;
    OZ_CUDA(cudaMemcpyAsync(visits, dv, nv * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(ns, dv + nv, (size_t)e->n_games * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

extern "C" int oz_search_get_root_stats(oz_engine* e, int32_t game, double* q, double* p, int32_t* qtag) {
    OZ_REQUIRE(e && q && p && qtag, "null argument");
    OZ_REQUIRE(game >= 0 && game < e->n_games, "game %d out of range", game);
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    double* dq = (double*)e->scratch;
    int* dt = (int*)(dq + 128);
    int rc = oz_tree_root_stats(e, game, dq, dq + 64, dt);
    if (rc) return rc;
    int found = -1;
    OZ_CUDA(cudaMemcpyAsync(q, dq, 64 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(p, dq + 64, 64 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(qtag, dt, 64 * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(&found, dt + 64, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    if (found < 0) { oz_set_error("root of game %d is not in the tree", game); return OZ_ERR_STATE; }
    return OZ_OK;
}

extern "C" int oz_search_get_status(oz_engine* e, int32_t* status) {
    OZ_REQUIRE(e && status, "null argument");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    OZ_CUDA(cudaMemcpyAsync(status, e->tp.status, (size_t)e->n_games * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

// ---- self-play --------------------------------------------------------------------------------------
extern "C" int oz_selfplay_begin(oz_engine* e, int32_t n_games, const uint64_t* black, const uint64_t* white,
                                 const int32_t* player, const uint64_t* game_ids, int32_t num_sims, double temperature,
                                 double e_greedy, int32_t max_moves) {
    OZ_REQUIRE(e, "null engine");
    OZ_REQUIRE(num_sims >= 2, "num_sims must be >= 2 (with 1 the reference's policy is all-zero, training.py:48-53)");
    OZ_REQUIRE(temperature >= 0.0, "temperature must be >= 0 (got %g)", temperature);
    OZ_REQUIRE(e_greedy >= 0.0 && e_greedy <= 1.0, "e_greedy must be in [0,1]");
    if (e->cfg.prior_mode == OZ_PRIOR_HOST) { oz_set_error("self-play needs OZ_PRIOR_HASH or OZ_PRIOR_NET"); return OZ_ERR_STATE; }
    OZ_REQUIRE(n_games >= 1, "n_games must be >= 1 (got %d)", n_games);
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    // more games than slots: the first max_games start now, the rest are queued and start as slots free up
    const int slots = n_games < e->cfg.max_games ? n_games : e->cfg.max_games;
    int rc = oz_tree_reserve_records(e, (size_t)n_games);
    if (rc) return rc;
    e->tp.leaf_count = e->leaf_count_base;  // leaf counters ping-pong between [0] and [4] (oz_selfplay_run); reset clears [0]
    e->tp.leaf_count_next = e->leaf_count_base + 4;
    rc = oz_tree_reset(e, slots, (const u64*)black, (const u64*)white, player, (const u64*)game_ids, true);
    if (rc) return rc;
    OzTreeParams& P = e->tp;
    e->search_started = false;
    P.q_black = P.q_white = nullptr; P.q_player = nullptr; P.q_ids = nullptr;
    if (black || player || game_ids) {  // staged for the whole job: validated below, and the queue reads them
        const size_t g8 = ((size_t)n_games * 8 + 255) & ~(size_t)255, g4 = ((size_t)n_games * 4 + 255) & ~(size_t)255;
        if (3 * g8 + g4 > e->q_bytes) {  // grow-only staging buffer
            if (e->q_buf) { OZ_CUDA(cudaStreamSynchronize(e->stream)); cudaFree(e->q_buf); e->q_buf = nullptr; e->q_bytes = 0; }
            cudaError_t qerr = cudaMalloc(&e->q_buf, 3 * g8 + g4);
            if (qerr != cudaSuccess) { oz_set_error("cudaMalloc for %d queued games failed: %s", n_games, cudaGetErrorString(qerr)); return OZ_ERR_NOMEM; }
            e->q_bytes = 3 * g8 + g4;
        }
        unsigned char* q = (unsigned char*)e->q_buf;
        if (black) {
            OZ_CUDA(cudaMemcpyAsync(q, black, (size_t)n_games * 8, cudaMemcpyHostToDevice, e->stream));
            OZ_CUDA(cudaMemcpyAsync(q + g8, white, (size_t)n_games * 8, cudaMemcpyHostToDevice, e->stream));
            P.q_black = (const u64*)q; P.q_white = (const u64*)(q + g8);
        }
        if (game_ids) {
            OZ_CUDA(cudaMemcpyAsync(q + 2 * g8, game_ids, (size_t)n_games * 8, cudaMemcpyHostToDevice, e->stream));
            P.q_ids = (const u64*)(q + 2 * g8);
        }
        if (player) {
            OZ_CUDA(cudaMemcpyAsync(q + 3 * g8, player, (size_t)n_games * 4, cudaMemcpyHostToDevice, e->stream));
            P.q_player = (const int*)(q + 3 * g8);
        }
    }
    if (black) {
        // a start whose side to move has no legal move would never reach a move transition (MCTS.simulate of a root
        // without actions): refuse the job instead of silently dropping the game
        int* bad = e->leaf_count_base + 3;
        e->h_pinned[6] = 0x7fffffff;
        OZ_CUDA(cudaMemcpyAsync(bad, &e->h_pinned[6], sizeof(int), cudaMemcpyHostToDevice, e->stream));
        validate_starts_kernel<<<(n_games + 255) / 256, 256, 0, e->stream>>>(n_games, P.q_black, P.q_white, P.q_player, P.full, bad);
        OZ_CUDA(cudaGetLastError());
        e->launches++;
        OZ_CUDA(cudaMemcpyAsync(&e->h_pinned[6], bad, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
        OZ_CUDA(cudaStreamSynchronize(e->stream));
        OZ_REQUIRE(e->h_pinned[6] == 0x7fffffff,
                   "start position %d is not playable (overlapping / off-board discs, or the side to move has no legal move)",
                   e->h_pinned[6]);
    }
    P.total_games = n_games;
    e->rec_games = n_games;
    OZ_CUDA(cudaMemsetAsync(P.leaf_count_next, 0, sizeof(int), e->stream));
    P.selfplay = 1;
    P.num_sims = num_sims;
    P.max_moves = max_moves;
    P.e_greedy = e_greedy;
    P.temperature = temperature;
    e->h_pinned[1] = slots;
    e->h_pinned[5] = slots;  // next queued game
    OZ_CUDA(cudaMemcpyAsync(P.n_active, &e->h_pinned[1], sizeof(int), cudaMemcpyHostToDevice, e->stream));
    OZ_CUDA(cudaMemcpyAsync(P.next_game, &e->h_pinned[5], sizeof(int), cudaMemcpyHostToDevice, e->stream));
    OZ_CUDA(cudaMemsetAsync(P.rec_action, 0xFF, (size_t)n_games * 64, e->stream));
    if (n_games > slots) {
        OZ_CUDA(cudaMemsetAsync(P.winner + slots, 0xFF, (size_t)(n_games - slots) * 4, e->stream));
        OZ_CUDA(cudaMemsetAsync(P.rec_nmoves + slots, 0, (size_t)(n_games - slots) * 4, e->stream));
    }
    search_begin_kernel<<<(P.G + 255) / 256, 256, 0, e->stream>>>(P, num_sims);
    OZ_CUDA(cudaGetLastError());
    e->launches++;
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    e->search_started = true;
    return OZ_OK;
}

extern "C" int oz_selfplay_run(oz_engine* e, int32_t steps, int32_t* n_active) {
    OZ_REQUIRE(e, "null engine");
    if (!e->search_started || !e->tp.selfplay) { oz_set_error("oz_selfplay_begin first"); return OZ_ERR_STATE; }
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    OzTreeParams& P = e->tp;
    const bool need_eval = e->cfg.prior_mode == OZ_PRIOR_NET || P.vl_width > 1;
    int active = -1;
    long long done = 0;
    u64 last_sims = ~0ull;
    u64* h_sims = (u64*)&e->h_pinned[8];
    while (steps < 0 || done < steps) {
        long long chunk = (steps < 0) ? 64 : (long long)steps - done;
        if (chunk > 64) chunk = 64;
        for (long long s = 0; s < chunk; ++s) {
            // leaf counters ping-pong between [0] and [4]: each tree launch clears the one the next launch will fill
            int rc = oz_tree_step(e);
            if (rc) return rc;
            if (need_eval && (rc = eval_leaves(e))) return rc;
            int* cur = P.leaf_count;
            P.leaf_count = P.leaf_count_next;
            P.leaf_count_next = cur;
        }
        done += chunk;
        OZ_CUDA(cudaMemcpyAsync(&e->h_pinned[2], P.n_active, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
        OZ_CUDA(cudaMemcpyAsync(h_sims, P.counters, sizeof(u64), cudaMemcpyDeviceToHost, e->stream));
        OZ_CUDA(cudaStreamSynchronize(e->stream));
        active = e->h_pinned[2];
        if (active <= 0) break;
        // a pool-exhausted game never finishes: report it instead of spinning forever
        if (steps < 0 && *h_sims == last_sims) {
            oz_set_error("self-play stalled with %d games active (node pool exhausted?)", active);
            return OZ_ERR_NOMEM;
        }
        last_sims = *h_sims;
    }
    if (active < 0) {
        OZ_CUDA(cudaMemcpyAsync(&e->h_pinned[2], P.n_active, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
        OZ_CUDA(cudaStreamSynchronize(e->stream));
        active = e->h_pinned[2];
    }
    if (n_active) *n_active = active;
    return OZ_OK;
}

extern "C" int oz_selfplay_get_records(oz_engine* e, uint64_t* rec_black, uint64_t* rec_white, uint8_t* rec_action,
                                       uint8_t* rec_player, int32_t* n_moves, int32_t* winner, int32_t* rec_visits) {
    OZ_REQUIRE(e && rec_black && rec_white && rec_action && rec_player && n_moves && winner, "null argument");
    OZ_REQUIRE(e->n_games > 0 && e->rec_games > 0, "no games");
    OZ_REQUIRE(!rec_visits || e->cfg.log_visits, "engine was created without log_visits");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    OzTreeParams& P = e->tp;
    size_t g = (size_t)e->rec_games;  // every game of the job, queued ones included
    OZ_CUDA(cudaMemcpyAsync(rec_black, P.rec_black, g * 64 * 8, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(rec_white, P.rec_white, g * 64 * 8, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(rec_action, P.rec_action, g * 64, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(rec_player, P.rec_player, g * 64, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(n_moves, P.rec_nmoves, g * 4, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(winner, P.winner, g * 4, cudaMemcpyDeviceToHost, e->stream));
    if (rec_visits) OZ_CUDA(cudaMemcpyAsync(rec_visits, P.rec_visits, g * 64 * 64 * 4, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

extern "C" int oz_selfplay_get_positions(oz_engine* e, uint64_t* black, uint64_t* white, int32_t* player) {
    OZ_REQUIRE(e, "null engine");
    OZ_REQUIRE(e->n_games > 0, "no games");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    size_t g = (size_t)e->n_games;
    if (black) OZ_CUDA(cudaMemcpyAsync(black, e->tp.black, g * 8, cudaMemcpyDeviceToHost, e->stream));
    if (white) OZ_CUDA(cudaMemcpyAsync(white, e->tp.white, g * 8, cudaMemcpyDeviceToHost, e->stream));
    if (player) OZ_CUDA(cudaMemcpyAsync(player, e->tp.player, g * 4, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

// ---- network ----------------------------------------------------------------------------------------
extern "C" int64_t oz_net_blob_floats(int32_t board_size, int32_t channels) {
    int size;  // the network depends on neither the rule set nor the scoring: both flags are accepted and ignored
    if (oz_decode_board(board_size, &size, nullptr)) return -1;
    return oz_net_blob_floats_impl(size, channels);
}

extern "C" int oz_net_load_weights(oz_engine* e, const float* blob, int64_t n_floats, int32_t channels) {
    OZ_REQUIRE(e && blob, "null argument");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    int rc = oz_tree_cache_clear(e);  // cached priors belong to the old weights
    if (rc) return rc;
    return oz_net_load(e, blob, n_floats, channels, false);
}

extern "C" int oz_net_load_weights_dev(oz_engine* e, const float* blob_dev, int64_t n_floats, int32_t channels) {
    OZ_REQUIRE(e && blob_dev, "null argument");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    int rc = oz_tree_cache_clear(e);
    if (rc) return rc;
    return oz_net_load(e, blob_dev, n_floats, channels, true);
}

extern "C" int oz_net_forward_dev(oz_engine* e, const uint64_t* own, const uint64_t* opp, int32_t n, float* pi,
                                  float* logits, float* v) {
    OZ_REQUIRE(e && own && opp && pi && v, "null argument");
    OZ_REQUIRE(n >= 1 && n <= e->max_leaves, "n %d out of range (capacity %d)", n, e->max_leaves);
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    e->h_pinned[3] = n;
    int* cnt = e->leaf_count_base + 1;
    OZ_CUDA(cudaMemcpyAsync(cnt, &e->h_pinned[3], sizeof(int), cudaMemcpyHostToDevice, e->stream));
    int rc = oz_net_forward(e, (const u64*)own, (const u64*)opp, cnt, n, pi, logits ? logits : e->leaf_logits, v);
    if (rc) return rc;
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

extern "C" int oz_net_forward_host(oz_engine* e, const uint64_t* own, const uint64_t* opp, int32_t n, float* pi,
                                   float* logits, float* v) {
    OZ_REQUIRE(e && own && opp && pi && v, "null argument");
    OZ_REQUIRE(n >= 1 && n <= e->max_leaves, "n %d out of range (capacity %d)", n, e->max_leaves);
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    const int nsq = e->tp.nsq;
    OZ_CUDA(cudaMemcpyAsync(e->tp.leaf_own, own, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
    OZ_CUDA(cudaMemcpyAsync(e->tp.leaf_opp, opp, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
    e->h_pinned[3] = n;
    int* cnt = e->leaf_count_base + 1;
    OZ_CUDA(cudaMemcpyAsync(cnt, &e->h_pinned[3], sizeof(int), cudaMemcpyHostToDevice, e->stream));
    int rc = oz_net_forward(e, e->tp.leaf_own, e->tp.leaf_opp, cnt, n, e->leaf_pi, e->leaf_logits, e->leaf_v);
    if (rc) return rc;
    // device rows have stride 64; host rows are N*N contiguous
    OZ_CUDA(cudaMemcpy2DAsync(pi, (size_t)nsq * 4, e->leaf_pi, 64 * 4, (size_t)nsq * 4, n, cudaMemcpyDeviceToHost, e->stream));
    if (logits)
        OZ_CUDA(cudaMemcpy2DAsync(logits, (size_t)nsq * 4, e->leaf_logits, 64 * 4, (size_t)nsq * 4, n, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(v, e->leaf_v, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

extern "C" int oz_net_layer_times(oz_engine* e, float* ms8) {
    OZ_REQUIRE(e && ms8, "null argument");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    return oz_net_times(e, ms8);
}

extern "C" int oz_net_set_timing(oz_engine* e, int32_t on) {
    OZ_REQUIRE(e, "null engine");
    oz_net_set_timing_impl(e, on != 0);
    return OZ_OK;
}

extern "C" int oz_net_get_activation(oz_engine* e, int32_t layer, void* host_bf16, int64_t bytes) {
    OZ_REQUIRE(e && host_bf16, "null argument");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    return oz_net_activation(e, layer, host_bf16, bytes);
}

extern "C" int oz_net_fp8_scales(oz_engine* e, float* out) {
    OZ_REQUIRE(e && out, "null argument");
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    return oz_net_scales(e, out);
}
