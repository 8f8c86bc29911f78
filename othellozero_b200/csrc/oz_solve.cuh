// oz_solve.cuh — the exact endgame search shared by the solver kernel (oz_solve.cu) and the tree kernel's leaf solver
// (oz_tree.cu): move ordering and the iterative fail-soft negamax.  DESIGN.md §12, §14.
#pragma once
#include "oz_engine.cuh"

constexpr int SOLVE_INF = 65;  // |margin| <= 64: (-65, 65) is the full window

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
// not negated).  Every level below the root places one disc, so a search from e empties suspends at most e - 1 levels:
// MAX_FRAMES bounds the empties of the positions a caller may search.
template <int RULES, int MAX_FRAMES = OZ_SOLVE_MAX_EMPTIES>
OZ_HD int solve_negamax(u64 own, u64 opp, u64 legal, int alpha, int beta, u64 full, u64 corners, u64 near_corners,
                             u64* nodes) {
    SolveFrame stack[MAX_FRAMES];
    int sp = 0;
    u64 moves = legal;
    int best = -SOLVE_INF - 1, neg = 0;
    u64 visited = 0;
    for (;;) {
        if (moves) {
            const u64 m = next_move(moves, corners, near_corners);
            moves ^= m;
            u64 o = own, p = opp, nl;
            const unsigned fl = ozbb::play_move<RULES>(m, &o, &p, full, &nl);
            ++visited;
            if (fl & ozbb::MOVE_FINISHED) {
                const int s = ozbb::popc(o) - ozbb::popc(p);  // o = the mover: the turn did not pass
                if (s > best) {
                    best = s;
                    if (s > alpha) { alpha = s; if (s >= beta) moves = 0; }
                }
                continue;
            }
            stack[sp++] = SolveFrame{own, opp, moves, pack_window(alpha, beta, best, neg)};
            const int sw = (fl & ozbb::MOVE_SWAPPED) ? 1 : 0;
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

// Corners and the squares next to them (C and X squares) of an N x N board, for next_move.
inline void oz_ordering_masks(int size, u64* corners, u64* near_corners) {
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
