// oz_bitboard.cuh — 64-bit bitboard statement of the reference's Othello rules.
//
// Bit index = r*8 + c for every board size N <= 8 (boards smaller than 8 live in the
// top-left N x N corner; squares outside are never set).  Ascending bit order ==
// the reference's row-major action order (np.argwhere, Othello/__init__.py:200-210).
//
// These are __host__ __device__ so the very same code is unit-tested on the CPU
// (tests/_bb_host.cpp) and runs inside the sm_100a kernels.
//
// Reference (relative to /root/reference):
//   legal moves   Othello/__init__.py:208-214   (identical to standard Othello)
//   flips         Othello/__init__.py:216-247   (NON-standard: no `break` after the
//                 bracketing own disc at :232-233 -> the walk continues through every
//                 occupied square and flips opponent discs beyond own discs too)
//   turn logic    Othello/__init__.py:147-159, othelo_mcts.py:43-49
//   terminal      Othello/__init__.py:249-252;  winner :254-260 (draw -> BLACK / ch0)
//
// Standard Othello flipping (a run of opponent discs flips only when the FIRST own disc beyond it brackets it) is
// offered next to the reference quirk: flip_mask_standard / flip_mask_standard_compact, and apply_move / play_move
// take the rule set as a template parameter (RULES_REFERENCE by default).  Legal moves, the initial position, the
// pass and terminal logic and the scoring are the same under both rule sets.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define OZ_HD __host__ __device__ __forceinline__
#else
#define OZ_HD static inline
#endif

typedef unsigned long long oz_u64;

namespace ozbb {

constexpr oz_u64 NOT_A = 0xFEFEFEFEFEFEFEFEull;  // clears column 0
constexpr oz_u64 NOT_H = 0x7F7F7F7F7F7F7F7Full;  // clears column 7
constexpr oz_u64 INNER = 0x7E7E7E7E7E7E7E7Eull;  // columns 1..6

OZ_HD int popc(oz_u64 x) {
#if defined(__CUDA_ARCH__)
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}
OZ_HD int msb_index(oz_u64 x) {  // x != 0
#if defined(__CUDA_ARCH__)
    return 63 - __clzll((long long)x);
#else
    return 63 - __builtin_clzll(x);
#endif
}

// All squares of an N x N board.
OZ_HD oz_u64 full_mask(int n) {
    oz_u64 row = (n >= 8) ? 0xFFull : ((1ull << n) - 1ull);
    oz_u64 m = 0;
    for (int r = 0; r < n; ++r) m |= row << (8 * r);
    return m;
}

// Initial position, Othello/__init__.py:177-184: WHITE on (p,p),(p+1,p+1); BLACK on the anti-diagonal.
OZ_HD void initial_position(int n, oz_u64* black, oz_u64* white) {
    int p = (n - 2) / 2;
    *white = (1ull << (p * 8 + p)) | (1ull << ((p + 1) * 8 + p + 1));
    *black = (1ull << (p * 8 + p + 1)) | (1ull << ((p + 1) * 8 + p));
}

// ---- legal moves --------------------------------------------------------------------
// One axis (both senses) of the classic bracketing scan, parallel-prefix form.
// `mo` = opponent discs that may sit strictly inside a bracket on this axis.
template <int D>
OZ_HD oz_u64 axis_moves(oz_u64 own, oz_u64 mo) {
    oz_u64 fl = mo & (own << D), fr = mo & (own >> D);
    fl |= mo & (fl << D);
    fr |= mo & (fr >> D);
    oz_u64 ml = mo & (mo << D), mr = mo & (mo >> D);
    fl |= ml & (fl << (2 * D));
    fr |= mr & (fr >> (2 * D));
    fl |= ml & (fl << (2 * D));
    fr |= mr & (fr >> (2 * D));
    return (fl << D) | (fr >> D);
}

// get_player_valid_actions as a mask (own = side to move).  `full` = full_mask(n).
OZ_HD oz_u64 legal_moves(oz_u64 own, oz_u64 opp, oz_u64 full) {
    oz_u64 mi = opp & INNER;
    oz_u64 m = axis_moves<1>(own, mi) | axis_moves<7>(own, mi) | axis_moves<9>(own, mi) | axis_moves<8>(own, opp);
    return m & full & ~(own | opp);
}

// ---- flips (reference quirk) -------------------------------------------------------------
// Occupied run starting at `gen` (0 or 1 bit) walking towards higher bits by step D,
// Kogge-Stone occluded fill; `pro` = occupied squares, pre-masked against column wrap.
template <int D>
OZ_HD oz_u64 fill_up(oz_u64 gen, oz_u64 pro) {
    gen |= pro & (gen << D);
    pro &= pro << D;
    gen |= pro & (gen << (2 * D));
    pro &= pro << (2 * D);
    gen |= pro & (gen << (4 * D));
    return gen;
}
template <int D>
OZ_HD oz_u64 fill_down(oz_u64 gen, oz_u64 pro) {
    gen |= pro & (gen >> D);
    pro &= pro >> D;
    gen |= pro & (gen >> (2 * D));
    pro &= pro >> (2 * D);
    gen |= pro & (gen >> (4 * D));
    return gen;
}

// Flips along +D: the contiguous occupied run behind the move, then every opponent disc that
// lies before the LAST own disc of that run (the reference keeps walking past own discs).
template <int D>
OZ_HD oz_u64 flips_up(oz_u64 m, oz_u64 own, oz_u64 opp, oz_u64 wrap) {
    oz_u64 occ = (own | opp) & wrap;
    oz_u64 first = (m << D) & wrap & opp;
    oz_u64 run = fill_up<D>(first, occ);
    oz_u64 anchors = run & own;
    if (!anchors) return 0;
    oz_u64 below = (1ull << msb_index(anchors)) - 1ull;
    return run & opp & below;
}
template <int D>
OZ_HD oz_u64 flips_down(oz_u64 m, oz_u64 own, oz_u64 opp, oz_u64 wrap) {
    oz_u64 occ = (own | opp) & wrap;
    oz_u64 first = (m >> D) & wrap & opp;
    oz_u64 run = fill_down<D>(first, occ);
    oz_u64 anchors = run & own;
    if (!anchors) return 0;
    oz_u64 lowest = anchors & (0ull - anchors);
    oz_u64 above = ~(lowest | (lowest - 1ull));
    return run & opp & above;
}

// get_action_flip_squares as a mask, for the move bit `m` (must be an empty square).
OZ_HD oz_u64 flip_mask(oz_u64 m, oz_u64 own, oz_u64 opp) {
    oz_u64 f = 0;
    f |= flips_up<1>(m, own, opp, NOT_A);     // (0,+1)
    f |= flips_up<9>(m, own, opp, NOT_A);     // (+1,+1)
    f |= flips_up<8>(m, own, opp, ~0ull);     // (+1,0)
    f |= flips_up<7>(m, own, opp, NOT_H);     // (+1,-1)
    f |= flips_down<1>(m, own, opp, NOT_H);   // (0,-1)
    f |= flips_down<9>(m, own, opp, NOT_H);   // (-1,-1)
    f |= flips_down<8>(m, own, opp, ~0ull);   // (-1,0)
    f |= flips_down<7>(m, own, opp, NOT_A);   // (-1,+1)
    return f;
}

// ---- flips (standard Othello) ----------------------------------------------------------------------------
// Along +D: the contiguous OPPONENT run behind the move (occluded fill through opponent discs only), kept iff the square
// right after it is an own disc.  `wrap` as in flips_up: shifting by D must not wrap across a column edge.
template <int D>
OZ_HD oz_u64 flips_up_standard(oz_u64 m, oz_u64 own, oz_u64 opp, oz_u64 wrap) {
    oz_u64 pro = opp & wrap;
    oz_u64 run = fill_up<D>((m << D) & pro, pro);
    return ((run << D) & wrap & own) ? run : 0ull;
}
template <int D>
OZ_HD oz_u64 flips_down_standard(oz_u64 m, oz_u64 own, oz_u64 opp, oz_u64 wrap) {
    oz_u64 pro = opp & wrap;
    oz_u64 run = fill_down<D>((m >> D) & pro, pro);
    return ((run >> D) & wrap & own) ? run : 0ull;
}

OZ_HD oz_u64 flip_mask_standard(oz_u64 m, oz_u64 own, oz_u64 opp) {
    oz_u64 f = 0;
    f |= flips_up_standard<1>(m, own, opp, NOT_A);
    f |= flips_up_standard<9>(m, own, opp, NOT_A);
    f |= flips_up_standard<8>(m, own, opp, ~0ull);
    f |= flips_up_standard<7>(m, own, opp, NOT_H);
    f |= flips_down_standard<1>(m, own, opp, NOT_H);
    f |= flips_down_standard<9>(m, own, opp, NOT_H);
    f |= flips_down_standard<8>(m, own, opp, ~0ull);
    f |= flips_down_standard<7>(m, own, opp, NOT_A);
    return f;
}

// Rule sets of apply_move / play_move (and of the kernels instantiated per rule set).
enum : int { RULES_REFERENCE = 0, RULES_STANDARD = 1 };

// ---- compact forms -------------------------------------------------------------------------------------
// The same arithmetic with the four axes walked by a loop with run-time shift counts (a 64-bit shift costs two
// instructions either way): about a quarter of the code.  For callers whose instruction FOOTPRINT matters more than
// their issue count - the tree kernel, whose hot path has to fit the 32 KB instruction cache (DESIGN 3d); the rules
// and perft kernels keep the unrolled templates.  tests/test_bitboard_host.py runs both forms over the golden vectors.
OZ_HD oz_u64 legal_moves_compact(oz_u64 own, oz_u64 opp, oz_u64 full) {
    const oz_u64 mi = opp & INNER;
    oz_u64 m = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int a = 0; a < 4; ++a) {
        const int D = (a == 0) ? 1 : 6 + a;  // 1, 7, 8, 9
        const oz_u64 mo = (D == 8) ? opp : mi;
        oz_u64 fl = mo & (own << D), fr = mo & (own >> D);
        fl |= mo & (fl << D);
        fr |= mo & (fr >> D);
        const oz_u64 ml = mo & (mo << D), mr = mo & (mo >> D);
        fl |= ml & (fl << (2 * D));
        fr |= mr & (fr >> (2 * D));
        fl |= ml & (fl << (2 * D));
        fr |= mr & (fr >> (2 * D));
        m |= (fl << D) | (fr >> D);
    }
    return m & full & ~(own | opp);
}

OZ_HD oz_u64 flip_mask_compact(oz_u64 m, oz_u64 own, oz_u64 opp) {
    const oz_u64 all = own | opp;
    oz_u64 f = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int a = 0; a < 4; ++a) {
        const int D = (a == 0) ? 1 : 6 + a;  // 1, 7, 8, 9
        // towards higher bits +1 / +9 must not wrap into column 0 and +7 not into column 7; mirrored going down
        const oz_u64 wu = (D == 8) ? ~0ull : (D == 7 ? NOT_H : NOT_A);
        const oz_u64 wd = (D == 8) ? ~0ull : (D == 7 ? NOT_A : NOT_H);
        {   // flips_up<D>
            oz_u64 pro = all & wu;
            oz_u64 gen = (m << D) & wu & opp;
            gen |= pro & (gen << D);
            pro &= pro << D;
            gen |= pro & (gen << (2 * D));
            pro &= pro << (2 * D);
            gen |= pro & (gen << (4 * D));
            const oz_u64 anchors = gen & own;
            const oz_u64 below = anchors ? (1ull << msb_index(anchors)) - 1ull : 0ull;
            f |= gen & opp & below;
        }
        {   // flips_down<D>
            oz_u64 pro = all & wd;
            oz_u64 gen = (m >> D) & wd & opp;
            gen |= pro & (gen >> D);
            pro &= pro >> D;
            gen |= pro & (gen >> (2 * D));
            pro &= pro >> (2 * D);
            gen |= pro & (gen >> (4 * D));
            const oz_u64 anchors = gen & own;
            const oz_u64 lowest = anchors & (0ull - anchors);
            const oz_u64 above = anchors ? ~(lowest | (lowest - 1ull)) : 0ull;
            f |= gen & opp & above;
        }
    }
    return f;
}

// flip_mask_standard in the compact form (same footprint constraints as flip_mask_compact).
OZ_HD oz_u64 flip_mask_standard_compact(oz_u64 m, oz_u64 own, oz_u64 opp) {
    oz_u64 f = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int a = 0; a < 4; ++a) {
        const int D = (a == 0) ? 1 : 6 + a;  // 1, 7, 8, 9
        const oz_u64 wu = (D == 8) ? ~0ull : (D == 7 ? NOT_H : NOT_A);
        const oz_u64 wd = (D == 8) ? ~0ull : (D == 7 ? NOT_A : NOT_H);
        {   // flips_up_standard<D>
            oz_u64 pro = opp & wu;
            oz_u64 gen = (m << D) & pro;
            gen |= pro & (gen << D);
            pro &= pro << D;
            gen |= pro & (gen << (2 * D));
            pro &= pro << (2 * D);
            gen |= pro & (gen << (4 * D));
            f |= ((gen << D) & wu & own) ? gen : 0ull;
        }
        {   // flips_down_standard<D>
            oz_u64 pro = opp & wd;
            oz_u64 gen = (m >> D) & pro;
            gen |= pro & (gen >> D);
            pro &= pro >> D;
            gen |= pro & (gen >> (2 * D));
            pro &= pro >> (2 * D);
            gen |= pro & (gen >> (4 * D));
            f |= ((gen >> D) & wd & own) ? gen : 0ull;
        }
    }
    return f;
}

// flip_board_squares, Othello/__init__.py:237-247: mover = own.
template <int RULES = RULES_REFERENCE>
OZ_HD void apply_move(oz_u64 m, oz_u64* own, oz_u64* opp) {
    oz_u64 f;
    if constexpr (RULES == RULES_STANDARD) f = flip_mask_standard(m, *own, *opp);
    else f = flip_mask(m, *own, *opp);
    *own |= f | m;
    *opp &= ~f;
}

// Outcome flags of a played move.
enum : unsigned { MOVE_SWAPPED = 1u, MOVE_PASSED = 2u, MOVE_FINISHED = 4u };

// Move + turn logic (OthelloGame.play :147-159 == get_next_state othelo_mcts.py:43-49).
// On return (*own,*opp) is in the frame of the side to move NEXT (swapped iff the opponent
// can move); *next_legal = that side's legal moves (0 iff finished).
template <int RULES = RULES_REFERENCE>
OZ_HD unsigned play_move(oz_u64 m, oz_u64* own, oz_u64* opp, oz_u64 full, oz_u64* next_legal) {
    apply_move<RULES>(m, own, opp);
    oz_u64 lo = legal_moves(*opp, *own, full);
    if (lo) {
        oz_u64 t = *own; *own = *opp; *opp = t;
        *next_legal = lo;
        return MOVE_SWAPPED;
    }
    oz_u64 lm = legal_moves(*own, *opp, full);
    *next_legal = lm;
    return lm ? MOVE_PASSED : MOVE_FINISHED;
}

// k-th (0-based) set bit of x, ascending. popc(x) > k.
OZ_HD int kth_set_bit(oz_u64 x, int k) {
    for (int i = 0; i < k; ++i) x &= x - 1ull;
#if defined(__CUDA_ARCH__)
    return __ffsll((long long)x) - 1;
#else
    return __builtin_ctzll(x);
#endif
}

// splitmix64 finaliser — the engine's counter-based RNG (SURVEY §8d config 2, Appendix B.3).
OZ_HD oz_u64 sm64(oz_u64 x) {
    x += 0x9E3779B97F4A7C15ull;
    oz_u64 z = x;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
OZ_HD unsigned pick_index(oz_u64 z, unsigned cnt) { return (unsigned)(((z >> 32) * (oz_u64)cnt) >> 32); }

// Key of a game's RNG stream.  Seed and game id are mixed NON-commutatively: with sm64(seed ^ id) the pair
// (seed 1, id g) replayed (seed 0, id g ^ 1), i.e. a different seed only permuted the same set of games.
OZ_HD oz_u64 stream_key(oz_u64 seed, oz_u64 id) { return sm64(sm64(seed) + id); }
// Self-play draws of move index p (training.py:48-56, othelo_mcts.py:54-62): value sm64(base + 4p + which).
constexpr oz_u64 EPISODE_STREAM = 0x5EEDC01Dull;
enum : unsigned { DRAW_COIN = 0u, DRAW_RANDOM_ACTION = 1u, DRAW_TIE_BREAK = 2u };
OZ_HD oz_u64 episode_key(oz_u64 seed, oz_u64 id) { return stream_key(seed ^ EPISODE_STREAM, id); }
OZ_HD oz_u64 episode_draw(oz_u64 base, int ply, unsigned which) { return sm64(base + 4ull * (oz_u64)ply + which); }

}  // namespace ozbb
