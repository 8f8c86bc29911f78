// oz_rules.cu — K1/K2/K3: one-thread-per-position bitboard rules kernels (sm_100a).
//
//   K1 rules_legal_kernel   get_player_valid_actions            Othello/__init__.py:208-214
//   K2 rules_apply_kernel   flip_board_squares + play turn logic Othello/__init__.py:237-247,147-159
//                           (== OthelloMCTS.get_next_state, othelo_mcts.py:43-49)
//   K3 perft_playout_kernel RandomOthelloAgent loop, whole game in registers   agents.py:20-24,71-84
//
// All three are integer-ALU bound: a position is 16 bytes in and 8-32 bytes out; the per-ply work is
// ~470 64-bit logical ops (DESIGN.md).  Coalesced 8-byte loads/stores, grid sized to fill 148 SMs.
#include <string.h>

#include "oz_engine.cuh"

using namespace ozbb;

__global__ void __launch_bounds__(256) rules_legal_kernel(const u64* __restrict__ own, const u64* __restrict__ opp,
                                                          u64* __restrict__ moves, long long n, u64 full) {
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        moves[i] = legal_moves(own[i], opp[i], full);
}

template <int RULES>
__global__ void __launch_bounds__(256)
rules_apply_kernel(const u64* __restrict__ own, const u64* __restrict__ opp, const int* __restrict__ sq,
                   u64* __restrict__ own_out, u64* __restrict__ opp_out, u32* __restrict__ flags,
                   u64* __restrict__ next_legal, long long n, u64 full) {
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        u64 o = own[i], p = opp[i];
        int s = sq[i];
        u64 m = (s >= 0 && s < 64) ? (1ull << s) : 0ull;
        u32 fl;
        u64 nl = 0;
        if (!(m & legal_moves(o, p, full))) {
            fl = 0x80000000u;  // not a legal move: position returned unchanged
        } else {
            fl = play_move<RULES>(m, &o, &p, full, &nl);
        }
        own_out[i] = o;
        opp_out[i] = p;
        flags[i] = fl;
        if (next_legal) next_legal[i] = nl;
    }
}

// get_board_players_points (Othello/__init__.py:258-260): popcount scoring.
__global__ void __launch_bounds__(256) rules_score_kernel(const u64* __restrict__ a, const u64* __restrict__ b,
                                                          int* __restrict__ ca, int* __restrict__ cb, long long n) {
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        ca[i] = popc(a[i]);
        cb[i] = popc(b[i]);
    }
}

// One thread = one whole random game; nothing but the final position touches memory.
template <int RULES>
__global__ void __launch_bounds__(256)
perft_playout_kernel(int n, u64 full, u64 seed, u64 first_id, long long n_games, int max_moves,
                     u64* __restrict__ black, u64* __restrict__ white, u32* __restrict__ info,
                     unsigned char* __restrict__ moves) {
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n_games; g += stride) {
        u64 own, opp;
        initial_position(n, &own, &opp);  // BLACK to move: own = black
        u32 player = 0, plies = 0, passes = 0, finished = 0;
        u64 base = stream_key(seed, first_id + (u64)g);
        u64 legal = legal_moves(own, opp, full);
        unsigned char* mv = moves ? moves + g * 64 : nullptr;
        while (legal && (max_moves < 0 || (int)plies < max_moves)) {
            u32 cnt = (u32)popc(legal);
            u32 k = pick_index(sm64(base + (u64)plies), cnt);
            int s = kth_set_bit(legal, (int)k);
            if (mv && plies < 64) mv[plies] = (unsigned char)s;
            u32 fl = play_move<RULES>(1ull << s, &own, &opp, full, &legal);
            ++plies;
            if (fl & MOVE_SWAPPED) player ^= 1u;
            if (fl & MOVE_PASSED) ++passes;
            if (fl & MOVE_FINISHED) finished = 1;
        }
        if (mv)
            for (u32 p = plies; p < 64; ++p) mv[p] = 0xFF;
        black[g] = player ? opp : own;
        white[g] = player ? own : opp;
        // OthelloGame.play switches current_player before it detects the end (Othello/__init__.py:147-156),
        // so a finished game reports the opponent of the last mover.
        if (finished) player ^= 1u;
        info[g] = plies | (player << 8) | (finished << 9) | (passes << 16);
    }
}

static int grid_for(long long n, int block) {
    long long b = (n + block - 1) / block;
    long long cap = 148LL * 8 * 4;  // 148 SMs x 8 resident 256-thread CTAs, a few waves
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

extern "C" int oz_rules_legal_moves_dev(int32_t board_size, const uint64_t* own, const uint64_t* opp,
                                        uint64_t* moves, int64_t n, void* stream) {
    int size;  // legal moves are the same under every rule set and scoring: the flags are accepted and ignored
    if (oz_decode_board(board_size, &size, nullptr)) return OZ_ERR_INVALID;
    if (n <= 0) return OZ_OK;
    rules_legal_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64*)own, (const u64*)opp,
                                                                            (u64*)moves, n, full_mask(size));
    OZ_CUDA(cudaGetLastError());
    return OZ_OK;
}

extern "C" int oz_rules_apply_dev(int32_t board_size, const uint64_t* own, const uint64_t* opp, const int32_t* sq,
                                  uint64_t* own_out, uint64_t* opp_out, uint32_t* flags, uint64_t* next_legal,
                                  int64_t n, void* stream) {
    int size, rules;
    if (oz_decode_board(board_size, &size, &rules)) return OZ_ERR_INVALID;
    if (n <= 0) return OZ_OK;
    auto kernel = rules == RULES_STANDARD ? rules_apply_kernel<RULES_STANDARD> : rules_apply_kernel<RULES_REFERENCE>;
    kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64*)own, (const u64*)opp, sq, (u64*)own_out,
                                                               (u64*)opp_out, flags, (u64*)next_legal, n, full_mask(size));
    OZ_CUDA(cudaGetLastError());
    return OZ_OK;
}

extern "C" int oz_rules_score_dev(const uint64_t* black, const uint64_t* white, int32_t* black_points,
                                  int32_t* white_points, int64_t n, void* stream) {
    if (n <= 0) return OZ_OK;
    rules_score_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64*)black, (const u64*)white,
                                                                           black_points, white_points, n);
    OZ_CUDA(cudaGetLastError());
    return OZ_OK;
}

extern "C" int oz_perft_playouts_dev(int32_t board_size, uint64_t seed, uint64_t first_game_id, int64_t n_games,
                                     int32_t max_moves, uint64_t* black, uint64_t* white, uint32_t* info,
                                     uint8_t* moves, void* stream) {
    int size, rules;
    if (oz_decode_board(board_size, &size, &rules)) return OZ_ERR_INVALID;
    if (n_games <= 0) return OZ_OK;
    // 128-thread CTAs: games end at different plies, smaller CTAs retire sooner (less tail per SM).
    long long blocks = (n_games + 127) / 128;
    long long cap = 148LL * 16 * 8;
    if (blocks > cap) blocks = cap;
    auto kernel = rules == RULES_STANDARD ? perft_playout_kernel<RULES_STANDARD> : perft_playout_kernel<RULES_REFERENCE>;
    kernel<<<(int)blocks, 128, 0, (cudaStream_t)stream>>>(size, full_mask(size), seed, first_game_id, n_games, max_moves,
                                                          (u64*)black, (u64*)white, info, moves);
    OZ_CUDA(cudaGetLastError());
    return OZ_OK;
}

// ---- host-buffer entry points (copies inside) ---------------------------------------------------------
// The reference calls the rules one position at a time from Python (Othello/__init__.py), so these calls are latency
// bound: each calling thread keeps ONE device scratch + ONE pinned staging buffer + ONE stream (grown on demand, reused
// across calls) instead of cudaMalloc/cudaFree per call; inputs go up in one async copy, outputs come back in one.
// One per calling thread, shared by every host-buffer entry point of the library (oz_engine.cuh).
OzHostScratch& oz_host_scratch() {
    static thread_local OzHostScratch s;
    return s;
}

extern "C" int oz_rules_legal_moves_host(int32_t device, int32_t board_size, const uint64_t* own,
                                         const uint64_t* opp, uint64_t* moves, int64_t n) {
    if (oz_decode_board(board_size, nullptr, nullptr)) return OZ_ERR_INVALID;
    OZ_REQUIRE(n >= 0 && (n == 0 || (own && opp && moves)), "null buffer");
    if (n == 0) return OZ_OK;
    OzHostScratch& S = oz_host_scratch();
    const size_t b8 = oz_up256((size_t)n * 8);
    int rc = S.reserve(device, 3 * b8);
    if (rc) return rc;
    memcpy(S.pin, own, (size_t)n * 8);
    memcpy(S.pin + b8, opp, (size_t)n * 8);
    OZ_CUDA(cudaMemcpyAsync(S.dev, S.pin, 2 * b8, cudaMemcpyHostToDevice, S.st));
    rc = oz_rules_legal_moves_dev(board_size, (const uint64_t*)S.dev, (const uint64_t*)(S.dev + b8),
                                  (uint64_t*)(S.dev + 2 * b8), n, S.st);
    if (rc) return rc;
    OZ_CUDA(cudaMemcpyAsync(S.pin + 2 * b8, S.dev + 2 * b8, (size_t)n * 8, cudaMemcpyDeviceToHost, S.st));
    OZ_CUDA(cudaStreamSynchronize(S.st));
    memcpy(moves, S.pin + 2 * b8, (size_t)n * 8);
    return OZ_OK;
}

extern "C" int oz_rules_apply_host(int32_t device, int32_t board_size, const uint64_t* own, const uint64_t* opp,
                                   const int32_t* sq, uint64_t* own_out, uint64_t* opp_out, uint32_t* flags,
                                   uint64_t* next_legal, int64_t n) {
    if (oz_decode_board(board_size, nullptr, nullptr)) return OZ_ERR_INVALID;
    OZ_REQUIRE(n >= 0 && (n == 0 || (own && opp && sq && own_out && opp_out && flags)), "null buffer");
    if (n == 0) return OZ_OK;
    OzHostScratch& S = oz_host_scratch();
    const size_t b8 = oz_up256((size_t)n * 8), b4 = oz_up256((size_t)n * 4);
    // layout: [own | opp | sq] inputs, [own' | opp' | next_legal | flags] outputs
    const size_t o_in = 0, o_out = 2 * b8 + b4, total = o_out + 3 * b8 + b4;
    int rc = S.reserve(device, total);
    if (rc) return rc;
    memcpy(S.pin, own, (size_t)n * 8);
    memcpy(S.pin + b8, opp, (size_t)n * 8);
    memcpy(S.pin + 2 * b8, sq, (size_t)n * 4);
    OZ_CUDA(cudaMemcpyAsync(S.dev + o_in, S.pin + o_in, o_out, cudaMemcpyHostToDevice, S.st));
    unsigned char* d = S.dev;
    rc = oz_rules_apply_dev(board_size, (const uint64_t*)d, (const uint64_t*)(d + b8), (const int32_t*)(d + 2 * b8),
                            (uint64_t*)(d + o_out), (uint64_t*)(d + o_out + b8), (uint32_t*)(d + o_out + 3 * b8),
                            (uint64_t*)(d + o_out + 2 * b8), n, S.st);
    if (rc) return rc;
    OZ_CUDA(cudaMemcpyAsync(S.pin + o_out, S.dev + o_out, 3 * b8 + b4, cudaMemcpyDeviceToHost, S.st));
    OZ_CUDA(cudaStreamSynchronize(S.st));
    memcpy(own_out, S.pin + o_out, (size_t)n * 8);
    memcpy(opp_out, S.pin + o_out + b8, (size_t)n * 8);
    if (next_legal) memcpy(next_legal, S.pin + o_out + 2 * b8, (size_t)n * 8);
    memcpy(flags, S.pin + o_out + 3 * b8, (size_t)n * 4);
    return OZ_OK;
}

extern "C" int oz_rules_score_host(int32_t device, const uint64_t* black, const uint64_t* white, int32_t* black_points,
                                   int32_t* white_points, int64_t n) {
    OZ_REQUIRE(n >= 0 && (n == 0 || (black && white && black_points && white_points)), "null buffer");
    if (n == 0) return OZ_OK;
    OzHostScratch& S = oz_host_scratch();
    const size_t b8 = oz_up256((size_t)n * 8), b4 = oz_up256((size_t)n * 4);
    int rc = S.reserve(device, 2 * b8 + 2 * b4);
    if (rc) return rc;
    memcpy(S.pin, black, (size_t)n * 8);
    memcpy(S.pin + b8, white, (size_t)n * 8);
    OZ_CUDA(cudaMemcpyAsync(S.dev, S.pin, 2 * b8, cudaMemcpyHostToDevice, S.st));
    rc = oz_rules_score_dev((const uint64_t*)S.dev, (const uint64_t*)(S.dev + b8), (int32_t*)(S.dev + 2 * b8),
                            (int32_t*)(S.dev + 2 * b8 + b4), n, S.st);
    if (rc) return rc;
    OZ_CUDA(cudaMemcpyAsync(S.pin + 2 * b8, S.dev + 2 * b8, 2 * b4, cudaMemcpyDeviceToHost, S.st));
    OZ_CUDA(cudaStreamSynchronize(S.st));
    memcpy(black_points, S.pin + 2 * b8, (size_t)n * 4);
    memcpy(white_points, S.pin + 2 * b8 + b4, (size_t)n * 4);
    return OZ_OK;
}

extern "C" int oz_perft_playouts_host(int32_t device, int32_t board_size, uint64_t seed, uint64_t first_game_id,
                                      int64_t n_games, int32_t max_moves, uint64_t* black, uint64_t* white,
                                      uint32_t* info, uint8_t* moves) {
    if (oz_decode_board(board_size, nullptr, nullptr)) return OZ_ERR_INVALID;
    OZ_REQUIRE(n_games >= 0 && (n_games == 0 || (black && white && info)), "null buffer");
    if (n_games == 0) return OZ_OK;
    OzHostScratch& S = oz_host_scratch();
    const size_t b8 = oz_up256((size_t)n_games * 8), b4 = oz_up256((size_t)n_games * 4);
    const size_t bm = moves ? oz_up256((size_t)n_games * 64) : 0;
    int rc = S.reserve(device, 2 * b8 + b4 + bm);
    if (rc) return rc;
    unsigned char* d = S.dev;
    rc = oz_perft_playouts_dev(board_size, seed, first_game_id, n_games, max_moves, (uint64_t*)d, (uint64_t*)(d + b8),
                               (uint32_t*)(d + 2 * b8), moves ? (uint8_t*)(d + 2 * b8 + b4) : nullptr, S.st);
    if (rc) return rc;
    OZ_CUDA(cudaMemcpyAsync(S.pin, S.dev, 2 * b8 + b4 + bm, cudaMemcpyDeviceToHost, S.st));
    OZ_CUDA(cudaStreamSynchronize(S.st));
    memcpy(black, S.pin, (size_t)n_games * 8);
    memcpy(white, S.pin + b8, (size_t)n_games * 8);
    memcpy(info, S.pin + 2 * b8, (size_t)n_games * 4);
    if (moves) memcpy(moves, S.pin + 2 * b8 + b4, (size_t)n_games * 64);
    return OZ_OK;
}


// ---- measurement aid: L2 read bandwidth ---------------------------------------------------------------------------------
// The table gather (oz_net.cu) is bound by the L2 -> SM path, so bench.py states its roofline against the L2 read
// bandwidth MEASURED on the box: every thread streams 16-byte loads (8 independent ones in flight) over an L2-resident
// buffer; the XOR of what it read is stored only if it matches a value it cannot have, which keeps the loads alive.
__global__ void __launch_bounds__(256) l2_read_probe_kernel(const uint4* __restrict__ buf, size_t n16, int passes, unsigned* sink) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    uint4 acc = make_uint4(0, 0, 0, 0);
    for (int p = 0; p < passes; ++p) {
        size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        for (; i + 7 * stride < n16; i += 8 * stride) {
            uint4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = __ldcg(buf + i + u * stride);  // .cg: L2 only, like a table row's first touch
#pragma unroll
            for (int u = 0; u < 8; ++u) { acc.x ^= v[u].x; acc.y ^= v[u].y; acc.z ^= v[u].z; acc.w ^= v[u].w; }
        }
        for (; i < n16; i += stride) { const uint4 v = __ldcg(buf + i); acc.x ^= v.x; acc.y ^= v.y; acc.z ^= v.z; acc.w ^= v.w; }
    }
    if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x9E3779B9u && passes < 0) *sink = acc.x;
}

extern "C" int oz_probe_l2_read(int32_t device, int32_t megabytes, int32_t passes, double* gb_per_s) {
    OZ_REQUIRE(gb_per_s && megabytes >= 1 && megabytes <= 4096 && passes >= 1, "bad argument");
    OZ_CUDA(cudaSetDevice(device));
    const size_t bytes = (size_t)megabytes << 20, n16 = bytes / 16;
    unsigned char* buf = nullptr;
    OZ_CUDA(cudaMalloc((void**)&buf, bytes + 16));
    struct Guard { void* p; cudaEvent_t a = nullptr, b = nullptr; ~Guard() { cudaFree(p); if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); } } g{buf};
    OZ_CUDA(cudaMemset(buf, 0x5A, bytes + 16));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    OZ_CUDA(cudaEventCreate(&g.a));
    OZ_CUDA(cudaEventCreate(&g.b));
    unsigned* sink = (unsigned*)(buf + bytes);
    l2_read_probe_kernel<<<sms * 8, 256>>>((const uint4*)buf, n16, 2, sink);  // warm: brings the buffer into L2
    OZ_CUDA(cudaEventRecord(g.a));
    l2_read_probe_kernel<<<sms * 8, 256>>>((const uint4*)buf, n16, passes, sink);
    OZ_CUDA(cudaEventRecord(g.b));
    OZ_CUDA(cudaEventSynchronize(g.b));
    OZ_CUDA(cudaGetLastError());
    float ms = 0.f;
    OZ_CUDA(cudaEventElapsedTime(&ms, g.a, g.b));
    *gb_per_s = (double)bytes * passes / (ms * 1e-3) / 1e9;
    return OZ_OK;
}
