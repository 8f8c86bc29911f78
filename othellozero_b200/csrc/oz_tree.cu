// oz_tree.cu — K4/K5/K6/K11: batched PUCT search over hash-keyed node pools in HBM (sm_100a).
//
// One WARP owns one game (its node arena, its transposition table, its root) and runs that game's
// simulations strictly one after another, exactly like the reference's recursive MCTS.simulate
// (MCTS/__init__.py:30-71) — that is what makes visit counts bit-exact.  Throughput comes from
// thousands of games (warps) in flight, not from parallelism inside a game.
//
//   select   lanes = children: coalesced loads of the node's P/Q/N rows, float64 UCB
//            Q + c*P*sqrt(Ns)/(1+N) (MCTS/__init__.py:168-170), warp arg-max with the reference's
//            first-max tie-break (:65)
//   frontier first traversal of an edge: bitboard move + pass/terminal test (othelo_mcts.py:43-49,
//            28-35), transposition lookup by exact board key (MCTS/__init__.py:42-44); the result
//            (child node / terminal value) is cached on the edge so later descents are pointer chases
//   expand   mask + normalise priors with numpy's pairwise np.sum order (MCTS/__init__.py:44-55,
//            othelo_mcts.py:69-80); one network evaluation per node (othelo_mcts.py:82-88)
//   backup   lanes = path entries; Q=(N*Q+v)/(N+1) with the reference's dynamic float32/float64 typing
//            (MCTS/__init__.py:68-71, SURVEY A.4), sign flip per ply
//   move     visit counts -> action (first arg-max or epsilon-random), example record, OthelloGame.play
//            (training.py:48-67)
//
// Virtual-loss waves (vl_width > 1, BASELINE configs[3]): the same warp runs up to vl_width descents per step, each
// leaving a virtual loss (an in-flight visit counted as a loss) on its path so that the next descent of the wave goes
// elsewhere; the leaves of a wave are evaluated together and backed up (virtual losses removed) in emission order at
// the start of the next step.  This fills the leaf batch with few games but changes visit counts relative to the
// sequential reference BY DESIGN; vl_width = 1 is the bit-exact mode and executes exactly the sequential code path.
// The in-flight count of an edge lives in the top 8 bits of its N word, the node's total in the header's `vns`.
#include "oz_engine.cuh"

using namespace ozbb;

#define FULLW 0xffffffffu
constexpr int TREE_WARPS = 4;  // warps (games) per CTA

// ---- node references -----------------------------------------------------------------------------------------------
// A node REFERENCE = (offset in 16-byte units << 6) | k, k = number of legal moves = number of child slots (<= 33).
// Carrying k in the reference lets a descent issue the loads of a node's header AND of its P/Q/N/child rows in ONE
// round (the row addresses depend on k): the pointer chase costs one memory latency per tree level instead of three
// (header -> rows -> child[best]).  Child words >= 0, path entries, root_node[] and table_find's result are references.
constexpr int REF_K_BITS = 6;
__device__ __forceinline__ int make_ref(u32 off, int k) { return (int)((off << REF_K_BITS) | (u32)k); }
__device__ __forceinline__ u32 ref_off(int ref) { return (u32)ref >> REF_K_BITS; }
__device__ __forceinline__ int ref_k(int ref) { return ref & ((1 << REF_K_BITS) - 1); }

__device__ __forceinline__ OzNodeHdr* node_at(unsigned char* arena, u32 off) {
    return (OzNodeHdr*)(arena + (size_t)off * 16);
}
__device__ __forceinline__ double* node_P(OzNodeHdr* h) { return (double*)((char*)h + sizeof(OzNodeHdr)); }
__device__ __forceinline__ double* node_Q(OzNodeHdr* h, int k) { return node_P(h) + k; }
__device__ __forceinline__ int* node_N(OzNodeHdr* h, int k) { return (int*)(node_P(h) + 2 * k); }
__device__ __forceinline__ int* node_child(OzNodeHdr* h, int k) { return node_N(h, k) + k; }
__host__ __device__ __forceinline__ u32 node_units(int k) { return (u32)((sizeof(OzNodeHdr) + 24 * k + 15) / 16); }

__device__ __forceinline__ u64 key_hash(u64 own, u64 opp) {
    u64 h = own * 0x9E3779B97F4A7C15ull ^ (opp + 0x632BE59BD9B4E019ull) * 0xC2B2AE3D27D4EB4Full;
    h ^= h >> 32;
    h *= 0xBF58476D1CE4E5B9ull;
    h ^= h >> 29;
    return h;
}

// The bulky scalar helpers are REAL calls with by-value arguments and a by-value result (nothing is passed by pointer,
// so no caller state is forced into local memory): every call site costs a few instructions instead of a few hundred,
// which is what keeps the kernel's hot loops inside the instruction cache (round 1: ~10.3 K SASS instructions, fetch
// stalls on top of the stall list).
// ... and they use the looped compact forms of oz_bitboard.cuh (a quarter of the unrolled templates' code, same issue count).
// The rule set and the scoring are template parameters of the kernel (one instantiation per combination, chosen at
// launch), never run-time branches, so the reference instantiations carry no cost for the standard variants
// (tools/sass_compare.py).
template <int RULES>
__device__ __noinline__ u64 flip_mask_call(u64 m, u64 own, u64 opp) {
    if constexpr (RULES == RULES_STANDARD) return flip_mask_standard_compact(m, own, opp);
    else return flip_mask_compact(m, own, opp);
}
__device__ __noinline__ u64 legal_moves_call(u64 own, u64 opp, u64 full) { return legal_moves_compact(own, opp, full); }

// play_move (oz_bitboard.cuh) over the out-of-line helpers.
template <int RULES>
__device__ __forceinline__ unsigned play_move_dev(u64 m, u64& own, u64& opp, u64 full, u64& next_legal) {
    const u64 f = flip_mask_call<RULES>(m, own, opp);
    own |= f | m;
    opp &= ~f;
    const u64 lo = legal_moves_call(opp, own, full);
    if (lo) {
        const u64 t = own; own = opp; opp = t;
        next_legal = lo;
        return MOVE_SWAPPED;
    }
    const u64 lm = legal_moves_call(own, opp, full);
    next_legal = lm;
    return lm ? MOVE_PASSED : MOVE_FINISHED;
}

// Warp-cooperative open-addressing lookup (32 slots per probe, one coalesced 256-byte load).
// Returns (insertion slot << 32) | (u32) reference; reference = -1 when the key is absent (the insertion slot is then
// where it would go, 0xffffffff if the table is full).
__device__ __noinline__ u64 table_find(const u64* __restrict__ table, int log2cap, unsigned char* arena, u64 own, u64 opp) {
    const int lane = threadIdx.x & 31;
    u64 h = key_hash(own, opp);
    u32 mask = (1u << log2cap) - 1u;
    u32 fp = (u32)(h >> 32);
    u32 start = (u32)h & mask;
#pragma unroll 1
    for (u32 w = 0; w <= mask; w += 32) {
        u32 idx = (start + w + (u32)lane) & mask;
        u64 ent = table[idx];
        unsigned empty = __ballot_sync(FULLW, ent == 0ull);
        unsigned cand = __ballot_sync(FULLW, ent != 0ull && (u32)(ent >> 32) == fp);
        if (empty) cand &= (1u << (__ffs(empty) - 1)) - 1u;
        while (cand) {
            int l = __ffs(cand) - 1;
            cand &= cand - 1u;
            u32 off = __shfl_sync(FULLW, (u32)ent, l) - 1u;
            OzNodeHdr* hd = node_at(arena, off);
            if (hd->own == own && hd->opp == opp) return (u64)(u32)make_ref(off, hd->k);
        }
        if (empty) return ((u64)((start + w + (u32)(__ffs(empty) - 1)) & mask) << 32) | 0xffffffffull;
    }
    return 0xffffffffffffffffull;
}
__device__ __forceinline__ int find_ref(u64 r) { return (int)(u32)r; }
__device__ __forceinline__ u32 find_ins(u64 r) { return (u32)(r >> 32); }

// Per-warp registers that describe the simulation in flight.
struct SimPath {
    u32 n0, e0, n1, e1;  // lane l holds path entries l and l+32 : (node reference, child slot)
};

__device__ __forceinline__ void path_set(SimPath& p, int lane, int depth, u32 node, u32 edge) {
    if (lane == (depth & 31)) {
        if (depth < 32) { p.n0 = node; p.e0 = edge; }
        else { p.n1 = node; p.e1 = edge; }
    }
}

// MCTS/__init__.py:68-70 for every edge of the path, lanes in parallel (a path never repeats a node).
// (is_int, iv, fv) = the value handed to the DEEPEST edge; it alternates sign going up (:71).
constexpr int N_MASK = 0x00FFFFFF;  // low 24 bits of an N word = visits, high 8 bits = virtual (in-flight) visits

__device__ __forceinline__ void backup_path(unsigned char* arena, const SimPath& p, int lane, int depth, bool is_int, int iv,
                                            float fv, bool vl) {
    for (int t = lane; t < depth; t += 32) {
        const int nref = (int)((t < 32) ? p.n0 : p.n1);
        u32 e = (t < 32) ? p.e0 : p.e1;
        bool neg = ((depth - 1 - t) & 1) != 0;
        int vi = neg ? -iv : iv;
        float vf = neg ? -fv : fv;
        OzNodeHdr* h = node_at(arena, ref_off(nref));
        const int k = ref_k(nref);  // no header round trip: Q/N addresses come from the reference
        double* Q = node_Q(h, k);
        int* N = node_N(h, k);
        const int nraw = N[e];
        double q = Q[e];
        const u64 qmask = h->qf32;
        const int nn = nraw & N_MASK;
        const int vn = (int)((unsigned)nraw >> 24);
        u64 bit = 1ull << e;
        bool f32 = (qmask & bit) != 0ull;
        if (nn == 0) {  // Q is python int 0
            if (is_int) {
                q = __ddiv_rn((double)(0 + vi), 1.0);
            } else {
                float s = __fadd_rn(0.0f, vf);
                q = (double)__fdiv_rn(s, 1.0f);
                f32 = true;
            }
        } else if (!f32) {  // python float
            double t64 = __dmul_rn((double)nn, q);
            if (is_int) {
                q = __ddiv_rn(__dadd_rn(t64, (double)vi), (double)(nn + 1));
            } else {
                float s = __fadd_rn(__double2float_rn(t64), vf);
                q = (double)__fdiv_rn(s, (float)(nn + 1));
                f32 = true;
            }
        } else {  // numpy float32
            float t32 = __fmul_rn((float)nn, (float)q);
            float s = __fadd_rn(t32, is_int ? (float)vi : vf);
            q = (double)__fdiv_rn(s, (float)(nn + 1));
        }
        Q[e] = q;
        N[e] = (nn + 1) | ((vl ? vn - 1 : vn) << 24);
        if (f32 && !(qmask & bit)) h->qf32 = qmask | bit;
        h->ns += 1;
        if (vl) h->vns -= 1;
    }
    __syncwarp();
}

// A descent of a virtual-loss wave that ran into a leaf already in flight: take its virtual losses back.
__device__ void revert_path(unsigned char* arena, const SimPath& p, int lane, int depth) {
    for (int t = lane; t < depth; t += 32) {
        const int nref = (int)((t < 32) ? p.n0 : p.n1);
        u32 e = (t < 32) ? p.e0 : p.e1;
        OzNodeHdr* h = node_at(arena, ref_off(nref));
        node_N(h, ref_k(nref))[e] -= (1 << 24);
        h->vns -= 1;
    }
    __syncwarp();
}

// Hash prior (SURVEY Appendix B.3) for one square / the value.
__device__ __forceinline__ float hash_pi(u64 key, int sq) {
    return (float)((double)((sm64(key + (u64)sq) >> 48) + 1ull) / 65536.0);
}
__device__ __forceinline__ float hash_v(u64 key) {
    return (float)(((double)(sm64(key ^ 0xABCDEFull) >> 48) - 32768.0) / 32768.0);
}

struct Pending {
    u64 own, opp, legal;
    int parent, pedge, depth;  // parent = reference of the parent node (-1: this leaf is the root)
};

// Expansion (MCTS/__init__.py:44-55) of `pd` with this lane's priors (pi_lo: square `lane`, pi_hi: square lane+32).
// Returns 1 = node created, 0 = the position already had a node (only inside a virtual-loss wave: two edges of the wave led
// to the same new position; this one just links to it), -1 = node pool / table exhausted.  The backup of -v is the caller's.
__device__ __forceinline__ int expand_node(const OzTreeParams& P, int slot, int lane, unsigned char* arena, u64* table,
                                           const Pending& pd, float pi_lo, float pi_hi, double* sa) {
    const int n = P.n, nsq = P.nsq;
    const int k = popc(pd.legal);
    const u32 units = node_units(k);
    const u32 off = P.bump[slot];
    const u64 fr = table_find(table, P.table_log2, arena, pd.own, pd.opp);
    const int found = find_ref(fr);
    const u32 ins = find_ins(fr);
    if (found >= 0) {
        if (lane == 0 && pd.parent >= 0) {
            OzNodeHdr* ph = node_at(arena, ref_off(pd.parent));
            node_child(ph, ref_k(pd.parent))[pd.pedge] = found;
        }
        __syncwarp();
        return 0;
    }
    if (((u64)off + units) * 16ull > P.arena_stride || ins == 0xffffffffu) return -1;

    // numpy order: a = pi(f32) * mask(f64) over the flat (N,N) array (othelo_mcts.py:69-73)
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        int sq = lane + 32 * half;
        int r = sq >> 3, c = sq & 7;
        if (r < n && c < n) {
            float pv = half ? pi_hi : pi_lo;
            sa[r * n + c] = ((pd.legal >> sq) & 1ull) ? (double)pv : 0.0;
        }
    }
    __syncwarp();
    // np.sum pairwise (8 strided accumulators, then a fixed tree, then the tail).  Rolled loops and the eight partial sums
    // exchanged through shared memory (sa[64..71]) instead of eight 64-bit shuffles: a tenth of the code, same additions.
    const int body = nsq - (nsq % 8);
    if (lane < 8) {
        double acc = sa[lane];
#pragma unroll 1
        for (int i = 8; i < body; i += 8) acc = __dadd_rn(acc, sa[i + lane]);
        sa[64 + lane] = acc;
    }
    __syncwarp();
    double sum = __dadd_rn(__dadd_rn(__dadd_rn(sa[64], sa[65]), __dadd_rn(sa[66], sa[67])),
                           __dadd_rn(__dadd_rn(sa[68], sa[69]), __dadd_rn(sa[70], sa[71])));
#pragma unroll 1
    for (int i = body; i < nsq; ++i) sum = __dadd_rn(sum, sa[i]);

    OzNodeHdr* h = node_at(arena, off);
    double* Pp = node_P(h);
    double* Qp = node_Q(h, k);
    int* Np = node_N(h, k);
    int* Cp = node_child(h, k);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        int sq = lane + 32 * half;
        if ((pd.legal >> sq) & 1ull) {
            int j = popc(pd.legal & ((1ull << sq) - 1ull));
            int r = sq >> 3, c = sq & 7;
            double pr = (sum > 0.0) ? __ddiv_rn(sa[r * n + c], sum) : __ddiv_rn(1.0, (double)k);
            Pp[j] = pr;
            Qp[j] = 0.0;
            Np[j] = 0;
            Cp[j] = OZ_CH_UNKNOWN;
        }
    }
    if (lane == 0) {
        h->own = pd.own; h->opp = pd.opp; h->legal = pd.legal; h->qf32 = 0ull;
        h->ns = 0; h->k = k; h->vns = 0; h->pad1 = 0;
        table[ins] = ((u64)(u32)(key_hash(pd.own, pd.opp) >> 32) << 32) | (u64)(off + 1u);
        P.bump[slot] = off + units;
        const int ref = make_ref(off, k);
        if (pd.parent >= 0) {
            OzNodeHdr* ph = node_at(arena, ref_off(pd.parent));
            node_child(ph, ref_k(pd.parent))[pd.pedge] = ref;
        } else {
            P.root_node[slot] = ref;
        }
    }
    __syncwarp();
    return 1;
}


// ---- cross-game evaluation cache -----------------------------------------------------------------------
// Identical positions give identical network outputs (the tower is row-independent), so one evaluation can
// serve every game that reaches the position — in the same step (ALIAS: share the leaf-batch row) or later
// (HIT: expand immediately from the cached priors, no network round trip).  Results are unchanged.
// 8-way buckets of 64-bit tags: [63:2] fingerprint | [1:0] state (0 empty, 1 claiming, 2 pending, 3 ready).
enum { CACHE_MISS = 0, CACHE_OWNER = 1, CACHE_ALIAS = 2, CACHE_HIT = 3 };

__device__ __forceinline__ u64 cache_hash(u64 own, u64 opp) {
    u64 h = (own ^ 0xD6E8FEB86659FD93ull) * 0x9E3779B97F4A7C15ull;
    h ^= h >> 31;
    h += opp * 0xC2B2AE3D27D4EB4Full;
    h ^= h >> 29;
    h *= 0x94D049BB133111EBull;
    h ^= h >> 32;
    return h;
}

__device__ __forceinline__ int cache_probe(const OzTreeParams& P, u64 own, u64 opp, int lane, u64* fp_out, int* cidx, int* leaf) {
    const u64 h = cache_hash(own, opp);
    const u64 fp = (h | (1ull << 63)) >> 2;  // 62 bits, never zero
    const u64 bucket = (h >> 3) & (((u64)1 << P.cache_log2_buckets) - 1ull);
    volatile u64* tags = (volatile u64*)P.cache_tags + bucket * 8;
    *fp_out = fp;
#pragma unroll 1
    for (int attempt = 0; attempt < 4096; ++attempt) {
        u64 t = (lane < 8) ? tags[lane] : 0ull;
        unsigned match = __ballot_sync(FULLW, lane < 8 && (t >> 2) == fp);
        unsigned empty = __ballot_sync(FULLW, lane < 8 && t == 0ull);
        if (match) {
            const int l = __ffs(match) - 1;
            const int st = (int)(__shfl_sync(FULLW, t, l) & 3ull);
            const int idx = (int)(bucket * 8) + l;
            if (st == 1) {  // another game is publishing this very position right now: wait for it
                __nanosleep(64);
                continue;
            }
            __threadfence();
            const volatile u64* key = (const volatile u64*)P.cache_keys + 2 * (size_t)idx;
            if (key[0] != own || key[1] != opp) return CACHE_MISS;  // fingerprint collision: evaluate uncached
            *cidx = idx;
            if (st == 3) return CACHE_HIT;
            *leaf = ((const volatile int*)P.cache_leaf)[idx];
            return CACHE_ALIAS;
        }
        if (!empty) return CACHE_MISS;  // bucket full
        const int l = __ffs(empty) - 1;
        u64 old = 0;
        if (lane == 0) old = atomicCAS((u64*)&tags[l], 0ull, (fp << 2) | 1ull);
        old = __shfl_sync(FULLW, old, 0);
        if (old == 0ull) {
            *cidx = (int)(bucket * 8) + l;
            return CACHE_OWNER;
        }
        // lost the race for this slot: look again (the winner may be the same position)
    }
    return CACHE_MISS;
}

// Publishing (copying an owner's priors into its entry and marking it ready) is the heads kernel's epilogue: oz_net.cu.

// Warp arg-max of (u, j): largest u, ties -> smallest j (the reference's first-max, MCTS/__init__.py:65); on return every
// lane holds the winning pair.  Doubles are mapped to 64-bit keys that order like the values, and the maximum is taken
// with three REDUX instructions (high word, low word among the high-word winners, smallest j among the winners) instead
// of five shuffle rounds of (2 SHFL + SHFL + 2 DSETP + 3 SEL): 50 -> 17 instructions on the hottest loop of the kernel.
__device__ __forceinline__ void warp_argmax(double& u, int& j) {
    const long long b = __double_as_longlong(__dadd_rn(u, 0.0));  // -0.0 -> +0.0: equal values, equal keys
    u32 hi = (u32)((unsigned long long)b >> 32), lo = (u32)b;
    const u32 neg = (u32)((int)hi >> 31);
    hi ^= neg | 0x80000000u;
    lo ^= neg;
    const u32 mh = __reduce_max_sync(FULLW, hi);
    const bool top = hi == mh;
    const u32 ml = __reduce_max_sync(FULLW, top ? lo : 0u);
    j = __reduce_min_sync(FULLW, (top && lo == ml) ? j : 0x7fffffff);
    const u32 back = (mh & 0x80000000u) ? 0u : 0xffffffffu;  // undo the key transform
    u = __longlong_as_double((long long)(((unsigned long long)((mh ^ 0x80000000u) ^ (back & 0x7fffffffu)) << 32) | (ml ^ back)));
}

// k-th (0-based) set bit of x by the whole (converged) warp: lane l ranks bits l and l+32.  Constant time, where the
// scalar loop (kth_set_bit) costs 4 instructions per skipped bit.
__device__ __forceinline__ int warp_kth_set_bit(u64 x, int k, int lane) {
    const u32 lo = (u32)x, hi = (u32)(x >> 32);
    const u32 below = (1u << lane) - 1u;
    const bool a = ((lo >> lane) & 1u) && __popc(lo & below) == k;
    const bool b = ((hi >> lane) & 1u) && __popc(lo) + __popc(hi & below) == k;
    const unsigned ba = __ballot_sync(FULLW, a), bb = __ballot_sync(FULLW, b);
    return ba ? __ffs(ba) - 1 : 31 + __ffs(bb);
}

// Global loads the compiler keeps where they are written (see the descent loop).
__device__ __forceinline__ int ld_i32(const int* p) {
    int v;
    asm volatile("ld.global.b32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ u64 ld_u64(const u64* p) {
    u64 v;
    asm volatile("ld.global.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_f64(const double* p) {
    double v;
    asm volatile("ld.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

// PUCT score of one edge (MCTS/__init__.py:168-170): Q + (c*P) * (sqrt(Ns) / (1 + N)) in float64, every operation rounded
// separately.  `nraw` = visits | in-flight << 24; an in-flight visit of a virtual-loss wave is scored as a loss.
__device__ __forceinline__ double ucb_value(int nraw, double q, double pj, double sq_ns, double c) {
    const int nj = nraw & N_MASK, vn = (int)((unsigned)nraw >> 24);
    if (vn) q = __ddiv_rn(__dadd_rn(__dmul_rn((double)nj, q), -(double)vn), (double)(nj + vn));
    const double bound = __ddiv_rn(sq_ns, (double)(1 + nj + vn));
    return __dadd_rn(q, __dmul_rn(__dmul_rn(c, pj), bound));
}
__device__ __noinline__ double ucb_value_call(int nraw, double q, double pj, double sq_ns, double c) {
    return ucb_value(nraw, q, pj, sq_ns, c);
}

// The engine step.  Every warp: (1) finishes the simulations that were waiting for their leaves, (2) keeps simulating
// until it needs another network evaluation or runs out of work.
//
// Structure (round 2): ONE loop whose body is either "expand the leaf at hand" or "run one descent", followed by ONE
// shared backup site.  Every heavy piece of code - expansion, backup, transposition lookup, move application - exists
// once in the kernel (round 1 had 3 inlined copies of the expansion, 5 of the backup, 3 of the lookup, 2 of play_move:
// 10.3 K SASS instructions, the instruction fetch was the top stall reason).
// 7 CTAs (28 warps) per SM = 72 registers: 148 x 28 = 4144 warps, so all 4096 games of configs[2] are still resident at
// once; at 8 CTAs / 64 registers the descent loop spilled and re-derived the arena pointer on every level.
#ifndef OZ_TREE_MIN_CTAS
#define OZ_TREE_MIN_CTAS 7
#endif
template <int RULES, int SCORING>
__global__ void __launch_bounds__(TREE_WARPS * 32, OZ_TREE_MIN_CTAS) tree_step_kernel(const OzTreeParams P) {
    __shared__ double s_a[TREE_WARPS][72];  // [0,64): masked priors of the node being expanded, [64,72): its partial sums
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int slot = blockIdx.x * TREE_WARPS + wib;
    if (slot >= P.G) return;
    double* sa = s_a[wib];

    // self-play ping-pongs two leaf counters: this launch fills P.leaf_count and clears the one the NEXT launch fills
    // (nobody reads it any more: the forward that consumed it ran before this launch) - no memset between steps
    if (P.leaf_count_next && blockIdx.x == 0 && threadIdx.x == 0) *P.leaf_count_next = 0;
    // the slot's state leaves in ONE round of loads (a launch typically runs one simulation per game, so the prologue's
    // dependent round trips are paid per simulation): everything is read before the status is looked at
    int status = ld_i32(P.status + slot);
    int sims_left = ld_i32(P.sims_left + slot);
    int gi = ld_i32(P.slot_game + slot);  // game index: where this episode's records go
    const int npend_raw = ld_i32(P.pend_count + slot);
    u64 black = ld_u64(P.black + slot), white = ld_u64(P.white + slot);
    int player = ld_i32(P.player + slot);
    int ply = ld_i32(P.ply + slot);
    if (status != OZ_GAME_ACTIVE && status != OZ_GAME_WAIT_LEAF) return;
    const long long t_start = clock64();

    unsigned char* arena = P.arena + (size_t)slot * P.arena_stride;
    u64* table = P.table + ((size_t)slot << P.table_log2);
    const int n = P.n;
    u64 c_sims = 0, c_nodes = 0, c_term = 0, c_trans = 0, c_moves = 0, c_hits = 0, c_alias = 0;
    int c_depth = 0;
    SimPath path{0, 0, 0, 0};
    Pending pd;

    const int V = P.vl_width;
    const bool vl = V > 1;
    // leaves parked by the previous launch, evaluated since: expanded first, in emission order (MCTS/__init__.py:44-57,67-71)
    const int npend = (status == OZ_GAME_WAIT_LEAF) ? npend_raw : 0;
    int next_pend = 0;
    status = OZ_GAME_ACTIVE;
    int inflight = 0;  // leaves parked by this launch (the current wave)


    // the leaf at hand: expanded by the next loop iteration.  src: 0 none, 1 priors in a global row, 2 closed-form hash priors
    int exp_src = 0;
    const float* exp_row = nullptr;
    float exp_v = 0.f;
    bool exp_counts_as_ran = false;

    int ran = 0;  // simulations completed by this launch without the evaluator
    while (true) {
        // values handed to the shared backup site at the end of the iteration
        bool do_backup = false, b_int = false;
        int b_iv = 0, b_depth = 0;
        float b_fv = 0.f;

        if (next_pend < npend || exp_src) {
            // ===== expansion site (the only one) =================================================================
            if (!exp_src) {
                const size_t pi_ = (size_t)slot * V + next_pend;
                ++next_pend;
                pd.own = P.pend_own[pi_]; pd.opp = P.pend_opp[pi_]; pd.legal = P.pend_legal[pi_];
                pd.parent = P.pend_parent[pi_]; pd.pedge = P.pend_edge[pi_]; pd.depth = P.pend_depth[pi_];
                const int li = P.pend_leaf[pi_];
                const u32* pn = P.path_node + pi_ * OZ_MAX_DEPTH;
                const u32* pe = P.path_edge + pi_ * OZ_MAX_DEPTH;
                if (lane < pd.depth) { path.n0 = pn[lane]; path.e0 = pe[lane]; }
                if (lane + 32 < pd.depth) { path.n1 = pn[lane + 32]; path.e1 = pe[lane + 32]; }
                // li >= 0: row of the evaluated leaf batch; li <= -2: evaluation-cache entry -(li+2) (wave mode parks hits too)
                exp_row = (li >= 0) ? P.leaf_pi + (size_t)li * 64 : P.cache_pi + (size_t)(-(li + 2)) * 64;
                exp_v = (li >= 0) ? P.leaf_v[li] : P.cache_v[-(li + 2)];
                exp_src = 1;
                exp_counts_as_ran = false;
            }
            // priors for this lane's two squares (row layout r*n+c with row stride 64)
            float pi_lo = 0.f, pi_hi = 0.f;
            if (exp_src == 1) {
                int r = lane >> 3, c = lane & 7;
                if (r < n && c < n) pi_lo = exp_row[r * n + c];
                r += 4;
                if (r < n && c < n) pi_hi = exp_row[r * n + c];
            } else {
                const u64 key = sm64(pd.own ^ sm64(pd.opp));
                pi_lo = hash_pi(key, lane); pi_hi = hash_pi(key, lane + 32);
                exp_v = hash_v(key);
            }
            exp_src = 0;
            const int made = expand_node(P, slot, lane, arena, table, pd, pi_lo, pi_hi, sa);
            if (made < 0) { status = OZ_GAME_POOL_FULL; break; }
            c_nodes += made; c_trans += 1 - made;
            if (exp_counts_as_ran) ++ran;
            do_backup = true; b_int = false; b_fv = -exp_v; b_depth = pd.depth;  // MCTS:57 returns -v to the parent
        } else {
            // yield (see oz_tree_alloc): a game that keeps finding evaluator-free simulations (terminal visits, cache hits)
            // stops once the launch has lasted `time_budget` clocks - by then the other games' warps have parked their
            // leaves and the evaluator is waiting - or after `sim_budget` of them; it resumes at the same simulation
            if (P.selfplay && ran > 0 &&
                ((P.sim_budget > 0 && ran >= P.sim_budget) || (P.time_budget > 0 && clock64() - t_start > P.time_budget))) {
                status = inflight > 0 ? OZ_GAME_WAIT_LEAF : OZ_GAME_ACTIVE;
                break;
            }
            if (sims_left - inflight <= 0) {
                if (inflight > 0) { status = OZ_GAME_WAIT_LEAF; break; }
                if (!P.selfplay) { status = OZ_GAME_IDLE; break; }
                // ---- move transition: training.py:45-67 --------------------------------------------------
                u64 own = player ? white : black, opp = player ? black : white;
                const int root = P.root_node[slot];
                OzNodeHdr* h = node_at(arena, ref_off(root));  // num_sims >= 2 guarantees the root exists
                const int k = ref_k(root);
                const u64 legal = h->legal;
                const int* Np = node_N(h, k);
                // visit counts by child slot; first arg-max == np.argwhere(policy == policy.max())[0]
                double best = -1.0; int bj = 1 << 20;
                for (int j = lane; j < k; j += 32) {
                    double cnt = (double)(Np[j] & N_MASK);
                    if (cnt > best) { best = cnt; bj = j; }
                }
                warp_argmax(best, bj);
                const u64 base = episode_key(P.seed, P.game_id[slot]);
                int aj = bj;
                if (P.temperature == 0.0) {
                    // othelo_mcts.py:54-62: the policy is one-hot on random.choice(arg-max set); a unique maximum needs no
                    // draw, ties are broken by the game's counter RNG over the tied actions in row-major order
                    const unsigned t0 = __ballot_sync(FULLW, lane < k && (double)(Np[lane] & N_MASK) == best);
                    const unsigned t1 = __ballot_sync(FULLW, lane + 32 < k && (double)(Np[lane + 32] & N_MASK) == best);
                    const u64 ties = (u64)t0 | ((u64)t1 << 32);
                    const int nt = popc(ties);
                    if (nt > 1) aj = warp_kth_set_bit(ties, (int)pick_index(episode_draw(base, ply, DRAW_TIE_BREAK), (u32)nt), lane);
                }
                const double coin = (double)(episode_draw(base, ply, DRAW_COIN) >> 11) * (1.0 / 9007199254740992.0);
                if (!(coin <= P.e_greedy)) aj = (int)pick_index(episode_draw(base, ply, DRAW_RANDOM_ACTION), (u32)k);
                const int sq = warp_kth_set_bit(legal, aj, lane);
                if (ply < 64) {
                    size_t ri = (size_t)gi * 64 + ply;
                    if (lane == 0) {
                        P.rec_black[ri] = black; P.rec_white[ri] = white;
                        P.rec_action[ri] = (unsigned char)sq; P.rec_player[ri] = (unsigned char)player;
                    }
                    if (P.log_visits) {
#pragma unroll
                        for (int half = 0; half < 2; ++half) {
                            int s = lane + 32 * half;
                            int cnt = ((legal >> s) & 1ull) ? (Np[popc(legal & ((1ull << s) - 1ull))] & N_MASK) : 0;
                            P.rec_visits[ri * 64 + s] = cnt;
                        }
                    }
                }
                u64 nl;
                const unsigned fl = play_move_dev<RULES>(1ull << sq, own, opp, P.full, nl);
                if (fl & MOVE_SWAPPED) player ^= 1;
                black = player ? opp : own;
                white = player ? own : opp;
                ++ply; ++c_moves;
                if (lane == 0) P.rec_nmoves[gi] = ply;
                const bool over = (fl & MOVE_FINISHED) != 0;
                if (over || (P.max_moves >= 0 && ply >= P.max_moves)) {
                    if (lane == 0) {
                        if constexpr (SCORING == SCORING_STANDARD) {
                            const int nb = popc(black), nw = popc(white);
                            P.winner[gi] = over ? (nb > nw ? 0 : (nb < nw ? 1 : OZ_WINNER_DRAW)) : -1;
                        } else {
                            P.winner[gi] = over ? ((popc(black) >= popc(white)) ? 0 : 1) : -1;
                        }
                        if (ply < 64) {  // entry n_moves of a game's record row = the position the episode ended in
                            P.rec_black[(size_t)gi * 64 + ply] = black; P.rec_white[(size_t)gi * 64 + ply] = white;
                        }
                    }
                    // the episode is over: take the next queued game into this slot, or retire the slot
                    int ng = P.total_games;
                    if (lane == 0) ng = atomicAdd(P.next_game, 1);
                    ng = __shfl_sync(FULLW, ng, 0);
                    if (ng >= P.total_games) {
                        status = OZ_GAME_FINISHED;
                        if (lane == 0) atomicSub(P.n_active, 1);
                        break;
                    }
                    gi = ng;
                    if (P.q_black) { black = P.q_black[ng]; white = P.q_white[ng]; }
                    else initial_position(n, &black, &white);
                    player = P.q_player ? P.q_player[ng] : 0;
                    ply = 0;
                    uint4* t4 = reinterpret_cast<uint4*>(table);  // a fresh tree: empty table, empty pool (training.py:30-32)
                    for (int i = lane; i < (1 << (P.table_log2 - 1)); i += 32) t4[i] = make_uint4(0, 0, 0, 0);
                    if (lane == 0) {
                        P.slot_game[slot] = ng;
                        P.game_id[slot] = P.q_ids ? P.q_ids[ng] : (u64)ng;
                        P.bump[slot] = 1;
                        P.root_node[slot] = -1;
                    }
                    __syncwarp();
                    sims_left = P.num_sims;
                    continue;
                }
                const int nr = find_ref(table_find(table, P.table_log2, arena, own, opp));
                if (lane == 0) P.root_node[slot] = nr;
                __syncwarp();
                sims_left = P.num_sims;
                continue;
            }

            if (inflight >= V) { status = OZ_GAME_WAIT_LEAF; break; }  // wave is full: wait for the evaluator

            // ---- one simulation: MCTS.simulate from the canonical root (othelo_mcts.py:22-26) -----------
            int node = P.root_node[slot];
            int depth = 0;
            int outcome = 0;  // 1 = terminal, 2 = leaf, 3 = ran into a leaf of this wave
            int term_val = 0;
            if (node < 0) {
                pd.own = player ? white : black;
                pd.opp = player ? black : white;
                pd.legal = legal_moves_call(pd.own, pd.opp, P.full);
                pd.parent = -1; pd.pedge = 0; pd.depth = 0;
                outcome = 2;
                if (!pd.legal) {  // a root whose side to move cannot move (search API only; self-play starts are validated)
                    status = P.selfplay ? OZ_GAME_FINISHED : OZ_GAME_IDLE;
                    if (P.selfplay && lane == 0) atomicSub(P.n_active, 1);
                    sims_left = 0;
                    break;
                }
            }
            while (!outcome) {
                OzNodeHdr* h = node_at(arena, ref_off(node));
                const int k = ref_k(node);
                const double* Pp = node_P(h);
                const double* Qp = node_Q(h, k);
                int* Np = node_N(h, k);
                int* Cp = node_child(h, k);
                // ONE round of loads per level: the header counters AND this lane's P/Q/N/child words (their addresses need
                // only the reference) are issued before anything is computed from them.  Round 1 read "ns" first and took its
                // square root before touching the rows - two dependent memory round trips per level.
                // (lanes beyond k re-read slot 0 - k >= 1 - so that the loads are unconditional and leave together.)
                // The loads are `asm volatile` so that the compiler neither sinks them into the branch that consumes them nor
                // starts the square root (which needs ns) ahead of them.
                const int jl = lane < k ? lane : 0;
                const int nraw0 = ld_i32(Np + jl);
                int c0 = ld_i32(Cp + jl), c1 = OZ_CH_UNKNOWN;
                const double q0 = ld_f64(Qp + jl), p0 = ld_f64(Pp + jl);
                const int ns = ld_i32(&h->ns);
                const int vns = ld_i32(&h->vns);
                const double sq_ns = __dsqrt_rn((double)(ns + vns));
                double bu = -1.0e300; int bj = 1 << 20;
                if (lane < k) { bu = ucb_value(nraw0, q0, p0, sq_ns, P.c); bj = lane; }
                if (k > 32 && lane + 32 < k) {  // more than 32 legal moves: a second candidate per lane (rare)
                    c1 = Cp[lane + 32];
                    const double u = ucb_value_call(Np[lane + 32], Qp[lane + 32], Pp[lane + 32], sq_ns, P.c);
                    if (u > bu) { bu = u; bj = lane + 32; }
                }
                warp_argmax(bu, bj);
                path_set(path, lane, depth, (u32)node, (u32)bj);
                ++depth;
                if (vl) {  // leave a virtual loss on the chosen edge for the rest of the wave
                    if (lane == 0) { Np[bj] += (1 << 24); h->vns = vns + 1; }
                    __syncwarp();
                }
                const int ch = __shfl_sync(FULLW, (bj < 32) ? c0 : c1, bj & 31);  // child[best] came with the same round
                if (ch >= 0) { node = ch; continue; }
                if (ch == OZ_CH_PENDING) { outcome = 3; break; }  // that leaf is already in flight in this wave
                if (ch == OZ_CH_TERM_NEG || ch == OZ_CH_TERM_POS) {
                    term_val = (ch == OZ_CH_TERM_POS) ? 1 : -1;
                    outcome = 1;
                    break;
                }
                if constexpr (SCORING == SCORING_STANDARD) {
                    if (ch == OZ_CH_TERM_DRAW) { term_val = 0; outcome = 1; break; }
                }
                // frontier: get_next_state (othelo_mcts.py:43-49)
                u64 own = h->own, opp = h->opp;
                const int sq = warp_kth_set_bit(h->legal, bj, lane);
                u64 nl;
                const unsigned fl = play_move_dev<RULES>(1ull << sq, own, opp, P.full, nl);
                if (fl & MOVE_FINISHED) {
                    // is_terminal_state -> return -reward; reward = +1 iff ch0 count >= ch1 count (draw -> BLACK)
                    if constexpr (SCORING == SCORING_STANDARD) {
                        // ... except that equal counts are a draw: reward 0, backed up as the integer 0
                        const int a = popc(own), b = popc(opp);
                        term_val = (a > b) ? -1 : (a < b ? 1 : 0);
                        if (lane == 0) Cp[bj] = (term_val > 0) ? OZ_CH_TERM_POS : (term_val < 0 ? OZ_CH_TERM_NEG : OZ_CH_TERM_DRAW);
                    } else {
                        int reward = (popc(own) >= popc(opp)) ? 1 : -1;
                        term_val = -reward;
                        if (lane == 0) Cp[bj] = (term_val > 0) ? OZ_CH_TERM_POS : OZ_CH_TERM_NEG;
                    }
                    outcome = 1;
                    break;
                }
                const int found = find_ref(table_find(table, P.table_log2, arena, own, opp));
                if (found >= 0) {  // transposition: the state already has a node
                    if (lane == 0) Cp[bj] = found;
                    ++c_trans;
                    node = found;
                    continue;
                }
                pd.own = own; pd.opp = opp; pd.legal = nl;
                pd.parent = node; pd.pedge = bj; pd.depth = depth;
                outcome = 2;
            }
            if (depth > c_depth) c_depth = depth;
            __syncwarp();

            if (outcome == 3) {
                revert_path(arena, path, lane, depth);
                status = OZ_GAME_WAIT_LEAF;  // inflight > 0 here: pending edges only exist inside a wave
                break;
            }
            if (outcome == 1) {
                ++c_term; ++ran;
                do_backup = true; b_int = true; b_iv = term_val; b_fv = (float)term_val; b_depth = depth;
            } else if (P.prior_mode == OZ_PRIOR_HASH && !vl) {
                exp_src = 2; exp_counts_as_ran = false;  // closed-form priors: expanded by the next iteration
                continue;
            } else {
                // hand the leaf to the evaluator and park this game (or reuse an evaluation of the same position)
                int li = -1, cidx = -1, cres = CACHE_MISS;
                u64 cfp = 0;
                if (P.cache_tags) {
                    cres = cache_probe(P, pd.own, pd.opp, lane, &cfp, &cidx, &li);
                    if (cres == CACHE_HIT) {
                        ++c_hits;
                        if (vl) {
                            li = -(cidx + 2);  // wave mode: keep the wave's composition independent of the cache - park the hit
                        } else {
                            exp_src = 1; exp_row = P.cache_pi + (size_t)cidx * 64; exp_v = P.cache_v[cidx];
                            exp_counts_as_ran = true;
                            continue;  // expanded by the next iteration, no network round trip
                        }
                    }
                }
                if (cres == CACHE_ALIAS) {
                    ++c_alias;
                } else if (li > -2) {
                    if (lane == 0) li = atomicAdd(P.leaf_count, 1);
                    li = __shfl_sync(FULLW, li, 0);
                    if (lane == 0) {
                        P.leaf_own[li] = pd.own; P.leaf_opp[li] = pd.opp;
                        if (P.cache_tags) P.leaf_cache_idx[li] = (cres == CACHE_OWNER) ? cidx : -1;
                        if (cres == CACHE_OWNER) {
                            P.cache_keys[2 * (size_t)cidx] = pd.own; P.cache_keys[2 * (size_t)cidx + 1] = pd.opp;
                            P.cache_leaf[cidx] = li;
                            __threadfence();
                            *((volatile u64*)P.cache_tags + cidx) = (cfp << 2) | 2ull;  // pending: same-step readers alias row li
                        }
                    }
                }
                {
                    const size_t pi_ = (size_t)slot * V + inflight;
                    if (lane == 0) {
                        P.pend_own[pi_] = pd.own; P.pend_opp[pi_] = pd.opp; P.pend_legal[pi_] = pd.legal;
                        P.pend_parent[pi_] = pd.parent; P.pend_edge[pi_] = pd.pedge; P.pend_depth[pi_] = pd.depth;
                        P.pend_leaf[pi_] = li;
                        if (vl && pd.parent >= 0) {  // later descents of this wave must not emit the same leaf again
                            OzNodeHdr* ph = node_at(arena, ref_off(pd.parent));
                            node_child(ph, ref_k(pd.parent))[pd.pedge] = OZ_CH_PENDING;
                        }
                    }
                    u32* pn = P.path_node + pi_ * OZ_MAX_DEPTH;
                    u32* pe = P.path_edge + pi_ * OZ_MAX_DEPTH;
                    if (lane < pd.depth) { pn[lane] = path.n0; pe[lane] = path.e0; }
                    if (lane + 32 < pd.depth) { pn[lane + 32] = path.n1; pe[lane + 32] = path.e1; }
                    __syncwarp();
                }
                ++inflight;
                if (pd.parent < 0) { status = OZ_GAME_WAIT_LEAF; break; }  // the root itself: nothing else can run before it exists
                continue;
            }
        }
        if (do_backup) {
            // ===== backup site (the only one): MCTS/__init__.py:67-71 ============================================
            backup_path(arena, path, lane, b_depth, b_int, b_iv, b_fv, vl);
            ++c_sims;
            --sims_left;
        }
    }

    if (lane == 0) {
        P.status[slot] = status;
        P.pend_count[slot] = inflight;
        P.sims_left[slot] = sims_left;
        P.black[slot] = black; P.white[slot] = white; P.player[slot] = player; P.ply[slot] = ply;
        if (c_sims) atomicAdd(&P.counters[0], c_sims);
        if (c_nodes) atomicAdd(&P.counters[1], c_nodes);
        if (c_term) atomicAdd(&P.counters[2], c_term);
        if (c_trans) atomicAdd(&P.counters[6], c_trans);
        if (c_hits) atomicAdd(&P.counters[3], c_hits);
        if (c_alias) atomicAdd(&P.counters[4], c_alias);
        if (c_moves) atomicAdd(&P.counters[7], c_moves);
        atomicMax(&P.counters[5], (u64)c_depth);
    }
}

// Wave mode with the closed-form priors: the "network" is this kernel, so that waves are formed exactly as with a
// real evaluator (leaves parked, evaluated together, expanded at the next step).
__global__ void hash_eval_kernel(const OzTreeParams P, float* __restrict__ pi, float* __restrict__ v) {
    const int lane = threadIdx.x & 31;
    const int li = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (li >= *P.leaf_count) return;
    const u64 key = sm64(P.leaf_own[li] ^ sm64(P.leaf_opp[li]));
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int sq = lane + 32 * half, r = sq >> 3, c = sq & 7;
        if (r < P.n && c < P.n) pi[(size_t)li * 64 + r * P.n + c] = hash_pi(key, sq);
    }
    if (lane == 0) v[li] = hash_v(key);
}

// MCTS.N(root, action) for every game (MCTS/__init__.py:73-84).
__global__ void tree_visits_kernel(const OzTreeParams P, int* __restrict__ visits, int* __restrict__ ns) {
    const int lane = threadIdx.x & 31;
    const int slot = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (slot >= P.G) return;
    unsigned char* arena = P.arena + (size_t)slot * P.arena_stride;
    const u64* table = P.table + ((size_t)slot << P.table_log2);
    int player = P.player[slot];
    u64 own = player ? P.white[slot] : P.black[slot], opp = player ? P.black[slot] : P.white[slot];
    const int root = find_ref(table_find(table, P.table_log2, arena, own, opp));
    int v0 = 0, v1 = 0, nsv = 0;
    if (root >= 0) {
        OzNodeHdr* h = node_at(arena, ref_off(root));
        u64 legal = h->legal;
        const int* Np = node_N(h, ref_k(root));
        if ((legal >> lane) & 1ull) v0 = Np[popc(legal & ((1ull << lane) - 1ull))] & N_MASK;
        if ((legal >> (lane + 32)) & 1ull) v1 = Np[popc(legal & ((1ull << (lane + 32)) - 1ull))] & N_MASK;
        nsv = h->ns | (h->vns << 24);  // vns must be 0 whenever no wave is in flight
    }
    visits[(size_t)slot * 64 + lane] = v0;
    visits[(size_t)slot * 64 + lane + 32] = v1;
    if (lane == 0) ns[slot] = nsv;
}

__global__ void tree_root_stats_kernel(const OzTreeParams P, int slot, double* __restrict__ q, double* __restrict__ p,
                                       int* __restrict__ tag, int* __restrict__ found) {
    const int lane = threadIdx.x & 31;
    unsigned char* arena = P.arena + (size_t)slot * P.arena_stride;
    const u64* table = P.table + ((size_t)slot << P.table_log2);
    int player = P.player[slot];
    u64 own = player ? P.white[slot] : P.black[slot], opp = player ? P.black[slot] : P.white[slot];
    const int root = find_ref(table_find(table, P.table_log2, arena, own, opp));
    if (lane == 0) *found = root;
    for (int half = 0; half < 2; ++half) {
        int s = lane + 32 * half;
        double qq = 0.0, pp = 0.0;
        int tt = -1;
        if (root >= 0) {
            OzNodeHdr* h = node_at(arena, ref_off(root));
            if ((h->legal >> s) & 1ull) {
                int j = popc(h->legal & ((1ull << s) - 1ull));
                int k = ref_k(root);
                qq = node_Q(h, k)[j];
                pp = node_P(h)[j];
                int nn = node_N(h, k)[j] & N_MASK;
                tt = (nn == 0) ? 0 : (((h->qf32 >> j) & 1ull) ? 2 : 1);
            }
        }
        q[s] = qq; p[s] = pp; tag[s] = tt;
    }
}

// ---- host side ---------------------------------------------------------------------------------------
int oz_tree_alloc(oz_engine* e) {
    const int G = e->cfg.max_games;
    OzTreeParams& P = e->tp;
    const int V = e->cfg.vl_width > 1 ? e->cfg.vl_width : 1;
    P.vl_width = V;
    // Endgame trees are mostly terminal edges: a game can run hundreds of simulations back to back without needing the
    // network while every other game waits for the launch to end (measured: 2 ms tree launches for ~1000 evaluations per
    // step over the last ten plies).  Bounding the run lets the step turn around; per-game results are unchanged (the
    // game resumes at the same simulation in the next launch).
    // Round 2: the count (8 in round 1) became a TIME budget.  In the steady-state mix of game phases a fixed count made the
    // endgame warps the tail of every launch (ncu: 98 us tree launches against ~30 us in the opening); bounding the launch
    // by time lets those games use exactly the slack the other warps leave (sweep in DESIGN.md 3d).
    const bool evaluator = e->cfg.prior_mode == OZ_PRIOR_NET || V > 1;
    // Wave mode keeps round 1's fixed COUNT: there a yield ends the wave, i.e. it decides which leaves share their virtual
    // losses, so it must not depend on timing (results stay reproducible and independent of the evaluation cache).
    P.sim_budget = evaluator ? (V > 1 ? 8 : 64) : 0;
    P.time_budget = (evaluator && V <= 1) ? 30000 : 0;  // SM clocks (~18 us at 1.65 GHz); 20-40 K measured equal, 5-10 K and 80 K slower
    if (const char* sb = getenv("OZ_TREE_SIM_BUDGET")) P.sim_budget = atoi(sb) > 0 ? atoi(sb) : 0;
    if (const char* tb = getenv("OZ_TREE_TIME_BUDGET")) P.time_budget = atoll(tb) > 0 ? atoll(tb) : 0;
    e->max_leaves = G * V;
    const size_t GV = (size_t)G * V;
    P.n = e->cfg.board_size;
    P.nsq = P.n * P.n;
    P.full = full_mask(P.n);
    P.prior_mode = e->cfg.prior_mode;
    P.log_visits = e->cfg.log_visits;
    P.c = e->cfg.c_puct;
    P.seed = e->cfg.seed;
    int log2 = 6;
    while ((1ll << log2) < 2ll * e->cfg.nodes_per_game) ++log2;
    e->table_log2 = log2;
    P.table_log2 = log2;
    // average node: 48 + 24*k bytes; k averages ~8.4 on 8x8 (max seen 20): budget 16 children per node
    u64 stride = (u64)e->cfg.nodes_per_game * (48 + 24 * 16);
    if (stride < 4096) stride = 4096;
    stride = (stride + 255) & ~255ull;
    // node references carry the offset (16-byte units) above REF_K_BITS bits of a positive int32
    OZ_REQUIRE(stride / 16 < (1ull << (31 - REF_K_BITS)), "nodes_per_game %d is too large for 32-bit node references",
               e->cfg.nodes_per_game);
    e->arena_stride = stride;
    P.arena_stride = stride;
    int rc = 0;
#define A(field, T, count) if ((rc = oz_dev_alloc<T>(e, (T**)&P.field, (size_t)(count)))) return rc;
    A(black, u64, G) A(white, u64, G) A(player, int, G) A(status, int, G) A(root_node, int, G)
    A(sims_left, int, G) A(ply, int, G) A(game_id, u64, G) A(slot_game, int, G)
    A(pend_own, u64, GV) A(pend_opp, u64, GV) A(pend_legal, u64, GV) A(pend_parent, int, GV) A(pend_edge, int, GV)
    A(pend_depth, int, GV) A(pend_leaf, int, GV) A(pend_count, int, G)
    A(path_node, u32, GV * OZ_MAX_DEPTH) A(path_edge, u32, GV * OZ_MAX_DEPTH)
    A(arena, unsigned char, (size_t)G * stride) A(bump, u32, G) A(table, u64, (size_t)G << log2)
    A(leaf_own, u64, GV) A(leaf_opp, u64, GV) A(leaf_count, int, 8)
    A(counters, u64, 8) A(n_active, int, 4)
    P.next_game = P.n_active + 1;
    P.total_games = 0;
    P.q_black = P.q_white = nullptr; P.q_player = nullptr; P.q_ids = nullptr;
    if ((rc = oz_tree_reserve_records(e, (size_t)G))) return rc;
    P.cache_tags = nullptr; P.cache_log2_buckets = 0;
    if (e->cfg.eval_cache_log2 > 0 && e->cfg.prior_mode == OZ_PRIOR_NET) {
        int lg = e->cfg.eval_cache_log2;
        if (lg < 10) lg = 10;
        if (lg > 28) lg = 28;
        const size_t entries = (size_t)1 << lg;
        A(cache_tags, u64, entries) A(cache_keys, u64, entries * 2) A(cache_leaf, int, entries)
        A(cache_pi, float, entries * 64) A(cache_v, float, entries) A(leaf_cache_idx, int, GV)
        P.cache_log2_buckets = lg - 3;
        e->cache_entries = entries;
        OZ_CUDA(cudaMemsetAsync(P.cache_tags, 0, entries * sizeof(u64), e->stream));
    }
#undef A
    e->scratch_bytes = GV * 64 * sizeof(float) + (size_t)G * 66 * sizeof(int) + 4096;  // put_priors / visits / reset staging
    if ((rc = oz_dev_alloc<unsigned char>(e, &e->scratch, e->scratch_bytes))) return rc;
    if ((rc = oz_dev_alloc<float>(e, &e->leaf_pi, GV * 64))) return rc;
    if ((rc = oz_dev_alloc<float>(e, &e->leaf_logits, GV * 64))) return rc;
    if ((rc = oz_dev_alloc<float>(e, &e->leaf_v, GV))) return rc;
    P.leaf_pi = e->leaf_pi;
    P.leaf_v = e->leaf_v;
    OZ_CUDA(cudaMemsetAsync(P.counters, 0, 8 * sizeof(u64), e->stream));
    OZ_CUDA(cudaMemsetAsync(P.status, 0, G * sizeof(int), e->stream));
    OZ_CUDA(cudaMemsetAsync(P.pend_count, 0, G * sizeof(int), e->stream));
    OZ_CUDA(cudaMemsetAsync(P.leaf_count, 0, 8 * sizeof(int), e->stream));
    e->leaf_count_base = P.leaf_count;
    P.leaf_count_next = nullptr;
    OZ_CUDA(cudaMemsetAsync(P.n_active, 0, 4 * sizeof(int), e->stream));
    return OZ_OK;
}

// Per-game record buffers (positions, actions, movers, visit counts, winner, plies): one allocation, regrown when a
// self-play job queues more games than the buffers hold.
int oz_tree_reserve_records(oz_engine* e, size_t games) {
    OzTreeParams& P = e->tp;
    if (games <= e->rec_capacity) return OZ_OK;
    if (e->rec_buf) { cudaStreamSynchronize(e->stream); cudaFree(e->rec_buf); e->rec_buf = nullptr; e->rec_capacity = 0; }
    const size_t per_game = 64 * 8 * 2 + 64 * 2 + 4 * 2 + (e->cfg.log_visits ? 64 * 64 * 4 : 0);
    unsigned char* q = nullptr;
    cudaError_t err = cudaMalloc((void**)&q, games * per_game + 256);
    if (err != cudaSuccess) {
        oz_set_error("cudaMalloc(%zu bytes) for %zu game records failed: %s", games * per_game, games, cudaGetErrorString(err));
        return OZ_ERR_NOMEM;
    }
    e->rec_buf = q;
    e->rec_capacity = games;
    P.rec_black = (u64*)q; q += games * 64 * 8;
    P.rec_white = (u64*)q; q += games * 64 * 8;
    P.rec_visits = nullptr;
    if (e->cfg.log_visits) { P.rec_visits = (int*)q; q += games * 64 * 64 * 4; }
    P.winner = (int*)q; q += games * 4;
    P.rec_nmoves = (int*)q; q += games * 4;
    P.rec_action = q; q += games * 64;
    P.rec_player = q;
    return OZ_OK;
}

__global__ void tree_init_slots_kernel(const OzTreeParams P, int n_games, const u64* __restrict__ black,
                                       const u64* __restrict__ white, const int* __restrict__ player,
                                       const u64* __restrict__ ids, int clear) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= P.G) return;
    if (g < n_games) {
        u64 b, w;
        if (black) { b = black[g]; w = white[g]; }
        else initial_position(P.n, &b, &w);
        P.black[g] = b; P.white[g] = w;
        P.player[g] = player ? player[g] : 0;
        if (clear) {
            P.game_id[g] = ids ? ids[g] : (u64)g;
            P.bump[g] = 1;  // offset 0 is never a node, so (off+1) != 0 and child >= 0 stays unambiguous
            P.ply[g] = 0;
            P.winner[g] = -1;
            P.rec_nmoves[g] = 0;
            P.slot_game[g] = g;
        }
        P.status[g] = OZ_GAME_IDLE;
        P.pend_count[g] = 0;
        P.root_node[g] = -1;
        P.sims_left[g] = 0;
    } else if (clear) {
        P.status[g] = OZ_GAME_IDLE;
        P.sims_left[g] = 0;
    }
}

// Re-resolve roots through the transposition table (after set_roots on a live tree).
__global__ void tree_find_roots_kernel(const OzTreeParams P) {
    const int lane = threadIdx.x & 31;
    const int slot = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (slot >= P.G) return;
    unsigned char* arena = P.arena + (size_t)slot * P.arena_stride;
    const u64* table = P.table + ((size_t)slot << P.table_log2);
    int player = P.player[slot];
    u64 own = player ? P.white[slot] : P.black[slot], opp = player ? P.black[slot] : P.white[slot];
    const int root = find_ref(table_find(table, P.table_log2, arena, own, opp));
    if (lane == 0) P.root_node[slot] = root;
}

int oz_tree_reset(oz_engine* e, int n_games, const u64* black, const u64* white, const int* player, const u64* ids,
                  bool clear) {
    OzTreeParams& P = e->tp;
    const int G = e->cfg.max_games;
    OZ_REQUIRE(n_games >= 1 && n_games <= G, "n_games %d out of range (max_games %d)", n_games, G);
    OZ_REQUIRE((black == nullptr) == (white == nullptr), "black/white must both be given or both NULL");
    u64 *d_b = nullptr, *d_w = nullptr, *d_id = nullptr;
    int* d_p = nullptr;
    // host start arrays are staged in the engine's persistent scratch: [black | white | ids | player], G entries each
    const size_t b8 = (size_t)n_games * 8, b4 = (size_t)n_games * 4, g8 = (size_t)G * 8;
    if (black) {
        d_b = (u64*)e->scratch; d_w = (u64*)(e->scratch + g8);
        OZ_CUDA(cudaMemcpyAsync(d_b, black, b8, cudaMemcpyHostToDevice, e->stream));
        OZ_CUDA(cudaMemcpyAsync(d_w, white, b8, cudaMemcpyHostToDevice, e->stream));
    }
    if (ids) {
        d_id = (u64*)(e->scratch + 2 * g8);
        OZ_CUDA(cudaMemcpyAsync(d_id, ids, b8, cudaMemcpyHostToDevice, e->stream));
    }
    if (player) {
        d_p = (int*)(e->scratch + 3 * g8);
        OZ_CUDA(cudaMemcpyAsync(d_p, player, b4, cudaMemcpyHostToDevice, e->stream));
    }
    if (clear) {
        OZ_CUDA(cudaMemsetAsync(P.table, 0, ((size_t)n_games << P.table_log2) * sizeof(u64), e->stream));
        OZ_CUDA(cudaMemsetAsync(P.counters, 0, 8 * sizeof(u64), e->stream));
        OZ_CUDA(cudaMemsetAsync(P.leaf_count, 0, sizeof(int), e->stream));
    }
    P.G = n_games;
    tree_init_slots_kernel<<<(G + 255) / 256, 256, 0, e->stream>>>(P, n_games, d_b, d_w, d_p, d_id, clear ? 1 : 0);
    OZ_CUDA(cudaGetLastError());
    e->launches++;
    if (!clear) {
        tree_find_roots_kernel<<<(n_games + 3) / 4, 128, 0, e->stream>>>(P);
        OZ_CUDA(cudaGetLastError());
        e->launches++;
    }
    e->n_games = n_games;
    return OZ_OK;
}

int oz_tree_step(oz_engine* e) {
    OzTreeParams& P = e->tp;
    int blocks = (P.G + TREE_WARPS - 1) / TREE_WARPS;
    auto kernel = e->rules == RULES_STANDARD
                      ? (e->scoring == SCORING_STANDARD ? tree_step_kernel<RULES_STANDARD, SCORING_STANDARD>
                                                        : tree_step_kernel<RULES_STANDARD, SCORING_REFERENCE>)
                      : (e->scoring == SCORING_STANDARD ? tree_step_kernel<RULES_REFERENCE, SCORING_STANDARD>
                                                        : tree_step_kernel<RULES_REFERENCE, SCORING_REFERENCE>);
    kernel<<<blocks, TREE_WARPS * 32, 0, e->stream>>>(P);
    OZ_CUDA(cudaGetLastError());
    e->launches++;
    return OZ_OK;
}

int oz_tree_visits(oz_engine* e, int* visits_dev, int* ns_dev) {
    OzTreeParams& P = e->tp;
    tree_visits_kernel<<<(P.G + 3) / 4, 128, 0, e->stream>>>(P, visits_dev, ns_dev);
    OZ_CUDA(cudaGetLastError());
    e->launches++;
    return OZ_OK;
}

int oz_tree_root_stats(oz_engine* e, int game, double* q_dev, double* p_dev, int* tag_dev) {
    OzTreeParams& P = e->tp;
    tree_root_stats_kernel<<<1, 32, 0, e->stream>>>(P, game, q_dev, p_dev, tag_dev, tag_dev + 64);
    OZ_CUDA(cudaGetLastError());
    e->launches++;
    return OZ_OK;
}

int oz_tree_cache_clear(oz_engine* e) {
    OzTreeParams& P = e->tp;
    if (!P.cache_tags) return OZ_OK;
    OZ_CUDA(cudaMemsetAsync(P.cache_tags, 0, e->cache_entries * sizeof(u64), e->stream));
    return OZ_OK;
}

int oz_tree_hash_eval(oz_engine* e) {
    OzTreeParams& P = e->tp;
    hash_eval_kernel<<<(P.G * P.vl_width + 7) / 8, 256, 0, e->stream>>>(P, e->leaf_pi, e->leaf_v);
    OZ_CUDA(cudaGetLastError());
    e->launches++;
    return OZ_OK;
}
