// Test-only host shim for the rule sets: compiles the product's __host__ __device__ bitboard header with g++ so that the
// standard flip forms, play_move<RULES> and a full-tree perft over it can be checked on the CPU (no GPU needed).
#include "../othellozero_b200/csrc/oz_bitboard.cuh"

// Full-tree perft over play_move<RULES>: a finished game is a leaf, a pass does not use up a ply.
template <int RULES>
static unsigned long long perft_rec(oz_u64 own, oz_u64 opp, oz_u64 legal, oz_u64 full, int depth) {
    if (depth == 0 || !legal) return 1;
    unsigned long long total = 0;
    for (oz_u64 l = legal; l; l &= l - 1) {
        oz_u64 o = own, p = opp, nl = 0;
        ozbb::play_move<RULES>(l & (0ull - l), &o, &p, full, &nl);
        total += perft_rec<RULES>(o, p, nl, full, depth - 1);
    }
    return total;
}

extern "C" {
unsigned long long bbr_legal(unsigned long long own, unsigned long long opp, int n) {
    return ozbb::legal_moves(own, opp, ozbb::full_mask(n));
}
unsigned long long bbr_flip_reference(int sq, unsigned long long own, unsigned long long opp) {
    return ozbb::flip_mask(1ull << sq, own, opp);
}
unsigned long long bbr_flip_standard(int sq, unsigned long long own, unsigned long long opp) {
    return ozbb::flip_mask_standard(1ull << sq, own, opp);
}
unsigned long long bbr_flip_standard_compact(int sq, unsigned long long own, unsigned long long opp) {
    return ozbb::flip_mask_standard_compact(1ull << sq, own, opp);
}
unsigned bbr_play(int standard, int sq, unsigned long long* own, unsigned long long* opp, int n,
                  unsigned long long* next_legal) {
    const oz_u64 full = ozbb::full_mask(n);
    return standard ? ozbb::play_move<ozbb::RULES_STANDARD>(1ull << sq, own, opp, full, next_legal)
                    : ozbb::play_move<ozbb::RULES_REFERENCE>(1ull << sq, own, opp, full, next_legal);
}
unsigned long long bbr_perft(int n, int depth, int standard) {
    oz_u64 own, opp, full = ozbb::full_mask(n);
    ozbb::initial_position(n, &own, &opp);
    oz_u64 legal = ozbb::legal_moves(own, opp, full);
    return standard ? perft_rec<ozbb::RULES_STANDARD>(own, opp, legal, full, depth)
                    : perft_rec<ozbb::RULES_REFERENCE>(own, opp, legal, full, depth);
}
void bbr_initial(int n, unsigned long long* b, unsigned long long* w) { ozbb::initial_position(n, b, w); }
}
