// oz_solve.cu — exact endgame solver: one thread per work item, iterative negamax alpha-beta (sm_100a).
//
// The value of a position is the final disc margin own - opp under perfect play by both sides, from the side to move
// (empties left at the end are not counted).  The game is the engine's: play_move<RULES> plays a move together with the
// automatic pass, and a position where neither side can move is finished.  The margin does not depend on the scoring:
// the W/D/L outcome under either scoring is a monotone function of it (engine.perfect_play_winner).  DESIGN.md §12.
//
//   solve_prepare_kernel   per position: empties, over-limit marking, item count per empties bucket
//   solve_scatter_kernel   work items in order of empties, most first (a counting sort over 21 buckets)
//   endgame_solve_kernel   persistent grid; each thread pulls items from one atomic counter and searches them
//   solve_finish_kernel    per-move mode: margin = max of the row; node counts out
#include <string.h>

#include "oz_engine.cuh"

using namespace ozbb;

constexpr int SOLVE_BUCKETS = OZ_SOLVE_MAX_EMPTIES + 1;
constexpr int SOLVE_INF = 65;          // |margin| <= 64: (-65, 65) is the full window
constexpr u64 WHOLE_POSITION = 0xFF;   // item low byte: search the position itself rather than one root move

// Device scratch of one call: [header | nodes_acc[n] | order[n * max(1, max_empties)]].
struct SolveHeader {
    unsigned long long hist[SOLVE_BUCKETS];    // items per empties bucket
    unsigned long long cursor[SOLVE_BUCKETS];  // items placed per bucket (scatter)
    unsigned long long next;                   // the work counter of the persistent grid
};

static size_t solve_scratch_bytes(long long n, int max_empties) {
    const long long per = max_empties > 1 ? max_empties : 1;  // a position has at most `empties` legal moves
    return oz_up256(sizeof(SolveHeader)) + oz_up256((size_t)n * 8) + oz_up256((size_t)n * per * 8);
}

OZ_HD int empties_of(u64 own, u64 opp, u64 full) { return popc(full & ~(own | opp)); }

// Items of a position in range: one per legal root move (per-move mode) or the whole position.
__device__ __forceinline__ int item_count(u64 own, u64 opp, u64 full, bool per_move) {
    const u64 legal = per_move ? legal_moves(own, opp, full) : 0;
    return legal ? popc(legal) : 1;
}

__global__ void __launch_bounds__(256)
solve_prepare_kernel(const u64* __restrict__ own, const u64* __restrict__ opp, long long n, u64 full, int max_empties,
                     bool per_move, signed char* __restrict__ margin, signed char* __restrict__ move_margin,
                     SolveHeader* __restrict__ hdr) {
    __shared__ unsigned long long hist[SOLVE_BUCKETS];
    for (int b = threadIdx.x; b < SOLVE_BUCKETS; b += blockDim.x) hist[b] = 0;
    __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const u64 o = own[i], p = opp[i];
        const int e = empties_of(o, p, full);
        if (move_margin) {
            uint4* row = (uint4*)(move_margin + i * 64);
            const unsigned none = 0x80808080u;  // OZ_SOLVE_NONE in every byte
            for (int k = 0; k < 4; ++k) row[k] = make_uint4(none, none, none, none);
        }
        if (e > max_empties) {
            margin[i] = (signed char)OZ_SOLVE_NONE;
            continue;
        }
        atomicAdd(&hist[e], (unsigned long long)item_count(o, p, full, per_move));
    }
    __syncthreads();
    for (int b = threadIdx.x; b < SOLVE_BUCKETS; b += blockDim.x)
        if (hist[b]) atomicAdd(&hdr->hist[b], hist[b]);
}

__global__ void __launch_bounds__(256)
solve_scatter_kernel(const u64* __restrict__ own, const u64* __restrict__ opp, long long n, u64 full, int max_empties,
                     bool per_move, SolveHeader* __restrict__ hdr, u64* __restrict__ order) {
    __shared__ unsigned long long base[SOLVE_BUCKETS];
    if (threadIdx.x == 0) {  // bucket e starts after every bucket with more empties
        unsigned long long s = 0;
        for (int e = OZ_SOLVE_MAX_EMPTIES; e >= 0; --e) { base[e] = s; s += hdr->hist[e]; }
    }
    __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const u64 o = own[i], p = opp[i];
        const int e = empties_of(o, p, full);
        if (e > max_empties) continue;
        u64 legal = per_move ? legal_moves(o, p, full) : 0;
        const int k = legal ? popc(legal) : 1;
        u64 slot = base[e] + atomicAdd(&hdr->cursor[e], (unsigned long long)k);
        if (!legal) {
            order[slot] = ((u64)i << 8) | WHOLE_POSITION;
            continue;
        }
        for (; legal; legal &= legal - 1) order[slot++] = ((u64)i << 8) | (u64)(__ffsll((long long)legal) - 1);
    }
}

// Static move ordering: corners first, squares next to a corner (C and X squares) last, everything else in between;
// ascending square order inside a class.  Results are exact whatever the order: it changes node counts only.
OZ_HD u64 next_move(u64 moves, u64 corners, u64 near_corners) {
    u64 c = moves & corners;
    if (!c) c = moves & ~near_corners;
    if (!c) c = moves;
    return c & (0ull - c);
}

// One suspended level of the search: the position, its moves not yet tried, and the window state (int8 each).
struct SolveFrame {
    u64 own, opp, moves;
    int packed;  // alpha | beta << 8 | best << 16 (bytes, two's complement) | negate << 24
};

OZ_HD int pack_window(int alpha, int beta, int best, int neg) {
    return (alpha & 0xFF) | ((beta & 0xFF) << 8) | ((best & 0xFF) << 16) | (neg << 24);
}

// Exact margin of (own, opp), own to move and own HAS a legal move `legal`, inside the window (alpha, beta), fail-soft.
// Iterative negamax: the current level lives in registers, suspended levels in a per-thread stack in local memory.
// A pass costs no level: play_move<RULES> returns MOVE_PASSED and the same side moves again in the child (its value is
// not negated).  Every level below the root places one disc, so a search from e empties suspends at most e - 1 levels.
template <int RULES>
OZ_HD int solve_negamax(u64 own, u64 opp, u64 legal, int alpha, int beta, u64 full, u64 corners, u64 near_corners,
                             u64* nodes) {
    SolveFrame stack[OZ_SOLVE_MAX_EMPTIES];
    int sp = 0;
    u64 moves = legal;
    int best = -SOLVE_INF - 1, neg = 0;
    u64 visited = 0;
    for (;;) {
        if (moves) {
            const u64 m = next_move(moves, corners, near_corners);
            moves ^= m;
            u64 o = own, p = opp, nl;
            const unsigned fl = play_move<RULES>(m, &o, &p, full, &nl);
            ++visited;
            if (fl & MOVE_FINISHED) {
                const int s = popc(o) - popc(p);  // o = the mover: the turn did not pass
                if (s > best) {
                    best = s;
                    if (s > alpha) { alpha = s; if (s >= beta) moves = 0; }
                }
                continue;
            }
            stack[sp++] = SolveFrame{own, opp, moves, pack_window(alpha, beta, best, neg)};
            const int sw = (fl & MOVE_SWAPPED) ? 1 : 0;
            const int a = sw ? -beta : alpha, b = sw ? -alpha : beta;
            own = o; opp = p; moves = nl;
            alpha = a; beta = b; best = -SOLVE_INF - 1; neg = sw;
            continue;
        }
        // every move of this level tried (or cut off): return `best` to the parent
        if (sp == 0) break;
        const int s = neg ? -best : best;
        const SolveFrame& f = stack[--sp];
        own = f.own; opp = f.opp; moves = f.moves;
        alpha = (signed char)(f.packed & 0xFF);
        beta = (signed char)((f.packed >> 8) & 0xFF);
        best = (signed char)((f.packed >> 16) & 0xFF);
        neg = (f.packed >> 24) & 1;
        if (s > best) {
            best = s;
            if (s > alpha) { alpha = s; if (s >= beta) moves = 0; }
        }
    }
    *nodes += visited;
    return best;
}

// Margin of a whole position (value mode, or a position without a legal move in per-move mode): a finished position is
// its disc difference; a mover without a move passes, and the position is worth minus the opponent's.
template <int RULES>
OZ_HD int solve_position(u64 own, u64 opp, u64 full, u64 corners, u64 near_corners, u64* nodes) {
    u64 legal = legal_moves(own, opp, full);
    int sign = 1;
    if (!legal) {
        const u64 lo = legal_moves(opp, own, full);
        if (!lo) return popc(own) - popc(opp);
        u64 t = own; own = opp; opp = t;
        legal = lo;
        sign = -1;
    }
    return sign * solve_negamax<RULES>(own, opp, legal, -SOLVE_INF, SOLVE_INF, full, corners, near_corners, nodes);
}

template <int RULES>
__global__ void __launch_bounds__(128)
endgame_solve_kernel(const u64* __restrict__ own, const u64* __restrict__ opp, const u64* __restrict__ order,
                     SolveHeader* __restrict__ hdr, u64 full, u64 corners, u64 near_corners,
                     signed char* __restrict__ margin, signed char* __restrict__ move_margin,
                     u64* __restrict__ nodes_acc) {
    unsigned long long total = 0;
    for (int e = 0; e <= OZ_SOLVE_MAX_EMPTIES; ++e) total += hdr->hist[e];
    for (;;) {
        const unsigned long long t = atomicAdd(&hdr->next, 1ull);
        if (t >= total) break;
        const u64 item = order[t];
        const long long i = (long long)(item >> 8);
        const int sq = (int)(item & 0xFF);
        const u64 o = own[i], p = opp[i];
        u64 nodes = 1;  // the item's root
        if (sq == (int)WHOLE_POSITION) {
            margin[i] = (signed char)solve_position<RULES>(o, p, full, corners, near_corners, &nodes);
        } else {
            // one root move searched with the full window; the item's root is the position after the move
            u64 co = o, cp = p, nl;
            const unsigned fl = play_move<RULES>(1ull << sq, &co, &cp, full, &nl);
            int v;
            if (fl & MOVE_FINISHED) v = popc(co) - popc(cp);
            else if (fl & MOVE_SWAPPED) v = -solve_negamax<RULES>(co, cp, nl, -SOLVE_INF, SOLVE_INF, full, corners, near_corners, &nodes);
            else v = solve_negamax<RULES>(co, cp, nl, -SOLVE_INF, SOLVE_INF, full, corners, near_corners, &nodes);
            move_margin[i * 64 + sq] = (signed char)v;
        }
        atomicAdd(&nodes_acc[i], (unsigned long long)nodes);
    }
}

__global__ void __launch_bounds__(256)
solve_finish_kernel(const u64* __restrict__ own, const u64* __restrict__ opp, long long n, u64 full, int max_empties,
                    signed char* __restrict__ margin, const signed char* __restrict__ move_margin,
                    const u64* __restrict__ nodes_acc, u64* __restrict__ nodes) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (nodes) nodes[i] = nodes_acc[i];
        if (!move_margin || empties_of(own[i], opp[i], full) > max_empties) continue;
        u64 legal = legal_moves(own[i], opp[i], full);
        if (!legal) continue;  // searched as a whole position
        int best = -SOLVE_INF - 1;
        for (; legal; legal &= legal - 1) {
            const int v = move_margin[i * 64 + __ffsll((long long)legal) - 1];
            best = v > best ? v : best;
        }
        margin[i] = (signed char)best;
    }
}

// Corners and the squares next to them (C and X squares) of an N x N board, for next_move.
static void ordering_masks(int size, u64* corners, u64* near_corners) {
    const int last = size - 1;
    const int cr[4] = {0, 0, last, last}, cc[4] = {0, last, 0, last};
    u64 c = 0, nc = 0;
    for (int k = 0; k < 4; ++k) {
        c |= 1ull << (cr[k] * 8 + cc[k]);
        for (int dr = -1; dr <= 1; ++dr)
            for (int dc = -1; dc <= 1; ++dc) {
                const int r = cr[k] + dr, col = cc[k] + dc;
                if (r >= 0 && r < size && col >= 0 && col < size) nc |= 1ull << (r * 8 + col);
            }
    }
    *corners = c;
    *near_corners = nc & ~c;
}

static int grid_for(long long n, int block) {
    long long b = (n + block - 1) / block;
    const long long cap = 148LL * 8 * 4;
    return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

// Argument checks shared by both entry points: every one of them fails before any CUDA call.
static int check_args(int32_t board_size, int* size, int* rules, const uint64_t* own, const uint64_t* opp, int64_t n,
               int32_t max_empties, const int8_t* margin) {
    if (oz_decode_board(board_size, size, rules)) return OZ_ERR_INVALID;
    OZ_REQUIRE(max_empties >= 0 && max_empties <= OZ_SOLVE_MAX_EMPTIES, "max_empties must be in [0, %d] (got %d)",
               OZ_SOLVE_MAX_EMPTIES, max_empties);
    OZ_REQUIRE(n >= 0 && n < (1LL << 55), "bad position count %lld", (long long)n);
    OZ_REQUIRE(n == 0 || (own && opp && margin), "null buffer");
    return OZ_OK;
}

// Every kernel of one call, on `st`; `scratch` holds solve_scratch_bytes(n, max_empties) bytes.
static int solve_launch(int size, int rules, const u64* own, const u64* opp, long long n, int max_empties, signed char* margin,
                 signed char* move_margin, u64* nodes, unsigned char* scratch, cudaStream_t st) {
    const u64 full = full_mask(size);
    const bool per_move = move_margin != nullptr;
    SolveHeader* hdr = (SolveHeader*)scratch;
    u64* nodes_acc = (u64*)(scratch + oz_up256(sizeof(SolveHeader)));
    u64* order = (u64*)(scratch + oz_up256(sizeof(SolveHeader)) + oz_up256((size_t)n * 8));
    OZ_CUDA(cudaMemsetAsync(scratch, 0, oz_up256(sizeof(SolveHeader)) + (size_t)n * 8, st));
    const int grid = grid_for(n, 256);
    solve_prepare_kernel<<<grid, 256, 0, st>>>(own, opp, n, full, max_empties, per_move, margin, move_margin, hdr);
    solve_scatter_kernel<<<grid, 256, 0, st>>>(own, opp, n, full, max_empties, per_move, hdr, order);
    u64 corners, near_corners;
    ordering_masks(size, &corners, &near_corners);
    auto kernel = rules == RULES_STANDARD ? endgame_solve_kernel<RULES_STANDARD> : endgame_solve_kernel<RULES_REFERENCE>;
    int dev = 0, sms = 148, per_sm = 1;
    OZ_CUDA(cudaGetDevice(&dev));
    OZ_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    OZ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 128, 0));
    // persistent: one resident wave (no more threads than items), each thread pulls items until none are left
    const long long items_max = n * (per_move && max_empties > 1 ? max_empties : 1);
    long long blocks = (long long)sms * (per_sm > 0 ? per_sm : 1);
    if (blocks > (items_max + 127) / 128) blocks = (items_max + 127) / 128;
    kernel<<<(int)(blocks > 0 ? blocks : 1), 128, 0, st>>>(own, opp, order, hdr, full, corners, near_corners, margin,
                                                            move_margin, nodes_acc);
    solve_finish_kernel<<<grid, 256, 0, st>>>(own, opp, n, full, max_empties, margin, move_margin, nodes_acc, nodes);
    OZ_CUDA(cudaGetLastError());
    return OZ_OK;
}

extern "C" int oz_endgame_solve_dev(int32_t board_size, const uint64_t* own, const uint64_t* opp, int64_t n,
                                    int32_t max_empties, int8_t* margin, int8_t* move_margin, uint64_t* nodes,
                                    void* stream) {
    int size, rules;
    int rc = check_args(board_size, &size, &rules, own, opp, n, max_empties, margin);
    if (rc || n == 0) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* scratch = nullptr;
    OZ_CUDA(cudaMallocAsync((void**)&scratch, solve_scratch_bytes(n, max_empties), st));
    rc = solve_launch(size, rules, (const u64*)own, (const u64*)opp, n, max_empties, (signed char*)margin,
                      (signed char*)move_margin, (u64*)nodes, scratch, st);
    cudaError_t e = cudaFreeAsync(scratch, st);
    if (rc) return rc;
    OZ_CUDA(e);
    return OZ_OK;
}

extern "C" int oz_endgame_solve_host(int32_t device, int32_t board_size, const uint64_t* own, const uint64_t* opp,
                                     int64_t n, int32_t max_empties, int8_t* margin, int8_t* move_margin,
                                     uint64_t* nodes) {
    int size, rules;
    int rc = check_args(board_size, &size, &rules, own, opp, n, max_empties, margin);
    if (rc || n == 0) return rc;
    const u64 full = full_mask(size);
    for (int64_t i = 0; i < n; ++i) {  // the device path does not validate content: do it here, before any launch
        OZ_REQUIRE(!(own[i] & opp[i]), "position %lld: own and opp discs overlap", (long long)i);
        OZ_REQUIRE(!((own[i] | opp[i]) & ~full), "position %lld: discs outside the %dx%d board", (long long)i, size, size);
        const int e = empties_of(own[i], opp[i], full);
        OZ_REQUIRE(e <= max_empties, "position %lld: %d empties > max_empties %d", (long long)i, e, max_empties);
    }
    OzHostScratch& S = oz_host_scratch();
    // layout: [own | opp] inputs, [margin | move_margin | nodes] outputs, then the solver's scratch
    const size_t b8 = oz_up256((size_t)n * 8), bm = oz_up256((size_t)n), brow = move_margin ? oz_up256((size_t)n * 64) : 0;
    const size_t o_out = 2 * b8, out_bytes = bm + brow + b8, o_scr = o_out + out_bytes;
    rc = S.reserve(device, o_scr + solve_scratch_bytes(n, max_empties));
    if (rc) return rc;
    memcpy(S.pin, own, (size_t)n * 8);
    memcpy(S.pin + b8, opp, (size_t)n * 8);
    OZ_CUDA(cudaMemcpyAsync(S.dev, S.pin, 2 * b8, cudaMemcpyHostToDevice, S.st));
    unsigned char* d = S.dev;
    rc = solve_launch(size, rules, (const u64*)d, (const u64*)(d + b8), n, max_empties, (signed char*)(d + o_out),
                      move_margin ? (signed char*)(d + o_out + bm) : nullptr, (u64*)(d + o_out + bm + brow), d + o_scr,
                      S.st);
    if (rc) return rc;
    OZ_CUDA(cudaMemcpyAsync(S.pin + o_out, S.dev + o_out, out_bytes, cudaMemcpyDeviceToHost, S.st));
    OZ_CUDA(cudaStreamSynchronize(S.st));
    memcpy(margin, S.pin + o_out, (size_t)n);
    if (move_margin) memcpy(move_margin, S.pin + o_out + bm, (size_t)n * 64);
    if (nodes) memcpy(nodes, S.pin + o_out + bm + brow, (size_t)n * 8);
    return OZ_OK;
}
