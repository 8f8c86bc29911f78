// oz_net.cu — K7..K10: the OthelloNNet policy/value tower (Net/OthelloNN.py:42-52) as bf16 tcgen05 kernels.
//
//   conv1 (Cin=2)     : the 3x3x2 binary input patch has only 3^9 = 19683 states, so conv1+BN+ReLU is a
//                       pre-computed 19683 x C bf16 table (built at weight load).
//   conv1∘conv2       : conv2 is linear in conv1's output, so tap t of conv2 applied to table row p is again a
//                       table: table2[p][t][:] (19683 x 9 x C bf16, built by the GEMM kernel at weight load) and
//                       the two layers are ONE gather-sum kernel (<= 9 row reads per output square), see
//                       conv2_table_gather_kernel.  OZ_NET_CONV2=gemm keeps conv1 = gather, conv2 = implicit GEMM.
//   conv3..4, fc1, fc2: ONE persistent, warp-specialised implicit-GEMM kernel:
//                       TMA (4-D tiled tensor map over the NHWC activation; taps = shifted boxes with
//                       hardware zero fill for padding='same') -> 128B-swizzled smem ring ->
//                       tcgen05.mma (128 x BLOCK_N x 16, bf16 in / fp32 accumulate in TMEM, double
//                       buffered) -> tcgen05.ld epilogue: + folded BN bias, ReLU, bf16 store.
//   heads             : same kernel, BLOCK_N = 128 (N^2 policy logits + 1 value row), epilogue = row
//                       softmax + tanh (Net/OthelloNN.py:50-52).  The net returns PROBABILITIES
//                       (NNetWrapper.predict, Net/NNet.py:85-87); logits are exposed for the parity check.
//
// BatchNormalization (eps 1e-3, moving statistics, Net/OthelloNN.py:43-49) is folded into the weights
// (fp32, then cast to bf16) and a per-channel fp32 bias at load time.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp8.h>
#include <stdlib.h>

#include <vector>

#include "oz_engine.cuh"

typedef __nv_bfloat16 bf16;

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 bf16 = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int STAGES = 4;
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;
constexpr int GEMM_THREADS = 256;
constexpr int EPI_RELU_BF16 = 0;
constexpr int EPI_HEADS = 1;
constexpr int EPI_LINEAR_BF16 = 2;  // no bias, no ReLU: builds the conv2 partial-product table
constexpr int N_PATTERNS = 19683;  // 3^9

struct GemmParams {
    int num_kb;          // K / 64
    int chunks_per_tap;  // Cin / 64 (conv) or num_kb (fc)
    int ntaps_x;         // 3 (conv) or 1 (fc)
    int pad;             // 1: padding='same', 0: 'valid' / fc
    int nb;              // boards per M tile (full-board box)
    int rows_per_board;  // OH*OW (1 for fc)
    int rows_valid;      // valid rows of an M tile (<= 128)
    // split tiles: when nb whole boards leave >= half a board of the 128 rows unused (36-row boards: 3 x 36 = 108),
    // an M tile is `halves` consecutive HALF boards (7 x 18 = 126 rows) fetched as one whole-board box + one half-board box
    int split;           // 0 / 1
    int halves;          // half-boards per tile (2*nb + 1)
    int half_rows;       // rows of a half board (OH/2 * OW)
    int half_h;          // OH / 2
    int tile_den;        // m_tiles = ceil(L * tile_num / tile_den): (1, nb) or (2, halves)
    int tile_num;
    int n_tiles;         // Nout / BLOCK_N
    int ldc;             // output row stride in elements
    int max_count;
    unsigned long long* trace;  // {min start ns, max end ns} of this launch, or null
    unsigned a_bytes;    // TMA bytes per A stage
    const int* count;    // device: number of boards in this batch
    const float* bias;   // [Nout] fp32 (BN folded)
    bf16* out;
    float* pi; float* logits; float* v;  // heads
    int nsq;
    // heads epilogue = also the evaluation cache's publish step (oz_tree.cu): row r of the batch belongs to cache entry
    // cache_idx[r] (>= 0) whose owner parked it as "pending"; null = no cache
    const int* cache_idx; float* cache_pi; float* cache_v; unsigned long long* cache_tags;
    const float* alpha;  // FP8 epilogues (oz_gemm2_kernel<OP_FP8_*>): out = relu(fma(acc, alpha[co], bias[co]))
};

// ---- PTX wrappers -------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (reported as a CUDA error) instead of hanging the GPU.  The bound is wall time
// (%globaltimer, looked at every 256 failed attempts), not a spin count: one try_wait may itself block for a
// hardware-defined time, and a count of 2^27 of those turned a mis-sized TMA transaction into a hang of minutes.
__device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
    unsigned long long t0 = 0;
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 255u) == 0) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t0 == 0) t0 = t;
            else if (t - t0 > 4000000000ull) __trap();  // 4 s: no kernel of the tower runs for more than a few ms
        }
    }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity);
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(m), "r"(bar), "r"(c0), "r"(c1) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// mbarrier arrives when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// Lean issue path: the MMA warp walks its loop converged and one ELECTED lane issues, which lets the compiler keep the
// descriptors, TMEM and barrier addresses in uniform registers (with `if (lane == 0)` it re-broadcasts every operand
// through an ELECT/R2UR loop, ~13 instructions per MMA: enough to pace an N=128 instruction at twice its pipe time).
// Descriptors are (low word, shared high word): only the start-address field in the low word changes between stages and
// k steps.
__device__ __forceinline__ bool elect_one() {  // one lane of the (converged) warp
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// Shared-memory matrix descriptor: K-major, 128-byte swizzle, 8-row groups 1024 bytes apart (SBO), Blackwell descriptor
// version bit; D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32.
constexpr uint32_t SW128_DESC_HI = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);  // SBO, version, SWIZZLE_128B
__device__ __forceinline__ uint32_t sw128_desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ void umma_bf16_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\t"
        "mov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(SW128_DESC_HI) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
// bf16x2 pack with the ReLU fused into the conversion (F2FP.RELU): low half = relu(lo), high half = relu(hi).
__device__ __forceinline__ uint32_t pack_relu_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// Programmatic dependent launch: let the next layer's CTAs start their prologue as ours retire, and make our own
// first read of the previous layer's output wait for that layer to have completed.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Instruction descriptor: D=f32, A=B=bf16, both K-major, M x N.
__host__ __device__ constexpr uint32_t make_idesc(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// kind::f8f6f4 instruction descriptor: D=f32, A=B=E4M3 (format code 0), both K-major, M x N.
__host__ __device__ constexpr uint32_t make_idesc_e4m3(int m, int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// Four e4m3 bytes (satfinite, round-to-nearest, ReLU fused: F2FP.SATFINITE.RELU.E4M3) from a..d, a in the lowest byte.
__device__ __forceinline__ uint32_t pack_relu_e4m3x4(float a, float b, float c, float d) {
    uint16_t lo, hi;
    asm("cvt.rn.satfinite.relu.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(b), "f"(a));
    asm("cvt.rn.satfinite.relu.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(d), "f"(c));
    return (uint32_t)lo | ((uint32_t)hi << 16);
}

// Table entries are consumed by fp32 accumulation only, so the pair (even, odd) is packed so that the odd element needs no
// extraction: the low half holds bf16_rn(even) as usual, and the high half is chosen such that the WHOLE 32-bit word, read
// as an fp32, is the representable value closest to `odd` (the low half then acts as 16 extra mantissa bits).  Candidates
// are 2^16 fp32-ulps apart, so |word - odd| <= half a bf16 ulp: the same bound as round-to-nearest bf16.
__device__ __forceinline__ uint32_t pack_pair_fused(float even, float odd) {
    const uint32_t lo = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(even));
    const uint32_t ob = __float_as_uint(odd);
    const uint32_t sign = ob & 0x80000000u;
    long long m = (long long)(ob & 0x7fffffffu) - (long long)lo + 32768;  // magnitudes order like integers
    if (m < 0) m = 0;
    uint32_t mag = ((uint32_t)m & 0xffff0000u) | lo;
    if (mag >= 0x7f800000u) mag = 0x7f7f0000u | lo;  // never round into inf/nan
    return sign | mag;
}

// Optional kernel timeline (OZ_NET_TRACE=<slots>): every CTA folds its start / end %globaltimer into the launch's slot;
// the table is printed to stderr when the engine is destroyed (tools/trace_forward.py).
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void trace_begin(unsigned long long* slot) {
    if (slot && threadIdx.x == 0) atomicMin(slot, global_ns());
}
__device__ __forceinline__ void trace_end(unsigned long long* slot) {
    if (slot && threadIdx.x == 0) atomicMax(slot + 1, global_ns());
}

template <int BLOCK_N>
struct GemmSmem {
    static constexpr int B_STAGE_BYTES = BLOCK_N * BLOCK_K * 2;
    static constexpr int OFF_A = 0;
    static constexpr int OFF_B = STAGES * A_STAGE_BYTES;
    static constexpr int OFF_BAR = OFF_B + STAGES * B_STAGE_BYTES;  // full[S], empty[S], tfull[2], tempty[2]
    static constexpr int OFF_TMEM = OFF_BAR + (2 * STAGES + 4) * 8;
    static constexpr int OFF_BIAS = OFF_TMEM + 16;                    // [2][BLOCK_N] floats
    static constexpr int BYTES = OFF_BIAS + 2 * BLOCK_N * 4;
    static constexpr int DYN_BYTES = BYTES + 1024;                    // manual 1024-byte alignment slack
};

template <int BLOCK_N, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
oz_gemm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapA2,
               const __grid_constant__ CUtensorMap mapB, const GemmParams p) {
    using S = GemmSmem<BLOCK_N>;
    constexpr int B_STAGE_BYTES = S::B_STAGE_BYTES;
    constexpr uint32_t TMEM_COLS = 2 * BLOCK_N;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gbase = smem_raw + (base - raw);
    const uint32_t sA = base + S::OFF_A, sB = base + S::OFF_B, sBar = base + S::OFF_BAR;
    auto full_bar = [&](int s) { return sBar + 8u * s; };
    auto empty_bar = [&](int s) { return sBar + 8u * (STAGES + s); };
    auto tfull_bar = [&](int a) { return sBar + 8u * (2 * STAGES + a); };
    auto tempty_bar = [&](int a) { return sBar + 8u * (2 * STAGES + 2 + a); };
    volatile uint32_t* s_tmem = (volatile uint32_t*)(gbase + S::OFF_TMEM);
    float* s_bias = (float*)(gbase + S::OFF_BIAS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    trace_begin(p.trace);
    int L = *p.count;
    if (L > p.max_count) L = p.max_count;
    const int m_tiles = (L * p.tile_num + p.tile_den - 1) / p.tile_den;
    const int num_tiles = m_tiles * p.n_tiles;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapB);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) {
        tmem_alloc(smem_u32((const void*)s_tmem), TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    pdl_launch_dependents();

    if (warp == 0) {
        {  // ===== TMA producer: converged warp, one elected lane issues (operands stay in uniform registers) =====
            pdl_wait();  // the activations we are about to read are the previous kernel's output
            // This one thread feeds the whole pipeline, so its per-stage instruction count is the supply rate: no integer
            // division in the k loop (taps and chunks are nested counters) and everything tile-invariant hoisted.  The
            // original `tap = kb / chunks_per_tap; ky = tap / ntaps_x` cost ~700 clk per stage against the 512 clk the
            // MMAs of a stage take (DESIGN 3c).
            int stage = 0; uint32_t phase = 0;
            const int ntaps_y = p.num_kb / (p.chunks_per_tap * p.ntaps_x);
            const uint32_t tx_bytes = p.a_bytes + (unsigned)B_STAGE_BYTES;
            const uint32_t off_main_after_half = (uint32_t)(p.half_rows * 128);
            const uint32_t off_half_after_main = (uint32_t)(p.nb * p.rows_per_board * 128);
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int m_tile = tile / p.n_tiles, n_idx = tile - m_tile * p.n_tiles;
                const int n0 = n_idx * BLOCK_N;
                // A boxes of this tile: (map, board, y offset, smem offset) x 2; the second is unused without split tiles
                const int hb0 = m_tile * p.halves;
                const bool odd = p.split && (hb0 & 1);
                const int bA = p.split ? ((hb0 >> 1) + (odd ? 1 : 0)) : m_tile * p.nb;      // whole-board box (mapA)
                const int bH = (hb0 >> 1) + (odd ? 0 : p.nb);                                  // half-board box (mapA2)
                const uint32_t offA = odd ? off_main_after_half : 0u;
                const uint32_t offH = odd ? 0u : off_half_after_main;
                const int yH = odd ? p.half_h : 0;
                int kcol = 0;
                for (int ky = -p.pad; ky < ntaps_y - p.pad; ++ky) {
                    for (int kx = -p.pad; kx < p.ntaps_x - p.pad; ++kx) {
                        for (int c0 = 0; c0 < p.chunks_per_tap * BLOCK_K; c0 += BLOCK_K) {
                            const uint32_t fb = full_bar(stage);
                            mbar_wait(empty_bar(stage), phase ^ 1u);
                            if (elect_one()) {
                                mbar_expect_tx(fb, tx_bytes);
                                const uint32_t dstA = sA + stage * A_STAGE_BYTES;
                                tma_load_4d(dstA + offA, &mapA, fb, c0, kx, ky, bA);
                                if (p.split) tma_load_4d(dstA + offH, &mapA2, fb, c0, kx, ky + yH, bH);
                                tma_load_2d(sB + stage * B_STAGE_BYTES, &mapB, fb, kcol, n0);
                            }
                            __syncwarp();
                            kcol += BLOCK_K;
                            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        {  // ===== MMA issuer: the warp walks the loop converged, one elected lane issues (see elect_one) =====
            constexpr uint32_t idesc = make_idesc(BLOCK_M, BLOCK_N);
            const uint32_t a_lo0 = sw128_desc_lo(sA), b_lo0 = sw128_desc_lo(sB);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                mbar_wait(tempty_bar(acc), acc_phase ^ 1u);  // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BLOCK_N);
                for (int kb = 0; kb < p.num_kb; ++kb) {
                    mbar_wait(full_bar(stage), phase);  // TMA bytes have landed
                    tc_fence_after();
                    const uint32_t a_lo = a_lo0 + (uint32_t)stage * (A_STAGE_BYTES >> 4);
                    const uint32_t b_lo = b_lo0 + (uint32_t)stage * (B_STAGE_BYTES >> 4);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BLOCK_K / UMMA_K; ++k)  // +2 = 32 bytes = 16 bf16 inside the 128-byte swizzle row
                            umma_bf16_lo(d_tmem, a_lo + 2u * k, b_lo + 2u * k, idesc, (kb | k) ? 1u : 0u);
                        umma_commit(empty_bar(stage));  // frees the smem stage once these MMAs retire
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
                if (elect_one()) umma_commit(tfull_bar(acc));  // accumulator complete -> epilogue
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> registers -> global =====
        const int ew = warp - 4;  // == warp % 4: TMEM lane quarter this warp may access
        const int et = threadIdx.x - 128;
        int acc = 0; uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int m_tile = tile / p.n_tiles, n_idx = tile - m_tile * p.n_tiles;
            float* bias = s_bias + acc * BLOCK_N;
            for (int i = et; i < BLOCK_N; i += 128) bias[i] = p.bias[n_idx * BLOCK_N + i];
            epi_bar_sync();
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
            const int r = ew * 32 + lane;
            const long long grow = (long long)m_tile * p.rows_valid + r;
            const bool ok = (r < p.rows_valid) && (grow < (long long)L * p.rows_per_board);
            const uint32_t t_row = tmem_base + (uint32_t)(acc * BLOCK_N) + ((uint32_t)(ew * 32) << 16);
            if constexpr (EPI == EPI_RELU_BF16 || EPI == EPI_LINEAR_BF16) {
                bf16* orow = p.out + grow * p.ldc + (long long)n_idx * BLOCK_N;
#pragma unroll 1
                for (int c = 0; c < BLOCK_N / 32; ++c) {
                    uint32_t v[32];
                    tmem_ld32(t_row + (uint32_t)(c * 32), v);
                    tmem_ld_wait();
                    if (ok) {
                        uint32_t packed[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float2 bj = *reinterpret_cast<const float2*>(bias + c * 32 + 2 * j);
                            const float2 y = __fadd2_rn(make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), bj);
                            if constexpr (EPI == EPI_LINEAR_BF16) packed[j] = pack_pair_fused(y.x, y.y);
                            else packed[j] = pack_relu_bf16x2(y.x, y.y);  // add.f32x2 + one F2FP.RELU per output pair
                        }
                        uint4* dst = reinterpret_cast<uint4*>(orow + c * 32);
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            dst[q] = make_uint4(packed[4 * q], packed[4 * q + 1], packed[4 * q + 2], packed[4 * q + 3]);
                    }
                }
            } else {
                // heads: columns [0,nsq) = policy logits, column nsq = value pre-activation
                float lg[96];
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    uint32_t v[32];
                    tmem_ld32(t_row + (uint32_t)(c * 32), v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) lg[c * 32 + j] = __uint_as_float(v[j]) + bias[c * 32 + j];
                }
                if (ok) {
                    const int nsq = p.nsq;
                    float mx = -3.0e38f;
#pragma unroll
                    for (int j = 0; j < 64; ++j) if (j < nsq) mx = fmaxf(mx, lg[j]);
                    float sum = 0.f;
                    float ex[64];
#pragma unroll
                    for (int j = 0; j < 64; ++j) { ex[j] = (j < nsq) ? expf(lg[j] - mx) : 0.f; sum += ex[j]; }
                    const float inv = 1.0f / sum;
                    float* prow = p.pi + grow * 64;
#pragma unroll
                    for (int j = 0; j < 64; j += 4)
                        *reinterpret_cast<float4*>(prow + j) = make_float4(ex[j] * inv, ex[j + 1] * inv, ex[j + 2] * inv, ex[j + 3] * inv);
                    if (p.logits) {  // only the parity / inspection entry points ask for the logits; self-play steps do not
                        float* lrow = p.logits + grow * 64;
#pragma unroll
                        for (int j = 0; j < 64; j += 4)
                            *reinterpret_cast<float4*>(lrow + j) = make_float4(lg[j], lg[j + 1], lg[j + 2], lg[j + 3]);
                    }
                    const float val = tanhf(nsq == 64 ? lg[64] : lg[36]);
                    p.v[grow] = val;
                    if (p.cache_idx) {
                        const int cidx = p.cache_idx[grow];
                        if (cidx >= 0) {  // this row's game owns a cache entry: fill it and mark it ready
                            float* crow = p.cache_pi + (size_t)cidx * 64;
#pragma unroll
                            for (int j = 0; j < 64; j += 4)
                                *reinterpret_cast<float4*>(crow + j) = make_float4(ex[j] * inv, ex[j + 1] * inv, ex[j + 2] * inv, ex[j + 3] * inv);
                            p.cache_v[cidx] = val;
                            // pending (2) -> ready (3): fire and forget.  No fence: nobody reads an entry's priors during this
                            // kernel (same-step readers share the leaf row), later kernels are ordered by the stream
                            atomicOr(p.cache_tags + cidx, 1ull);
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(acc));
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
    trace_end(p.trace);
}

// ---- 2-CTA variant: cta_group::2, one 256 x 256 accumulator tile per SM pair ---------------------------------
// Each CTA of the pair stages its own 128 rows of A and its own 128-row half of the B tile (32 KB per k-block instead
// of 48 KB: a third less L2->SMEM traffic and half the B operand reads per SM), which also buys a 6-deep ring.  The
// leader CTA issues tcgen05.mma.cta_group::2 for both; completion is multicast to the barriers of both CTAs.
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(m), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\t"
        "mov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(SW128_DESC_HI) : "memory");
}
__device__ __forceinline__ void umma_e4m3_2sm_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\t"
        "mov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], da, db, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(SW128_DESC_HI) : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(cta_mask) : "memory");
}

constexpr int STAGES2 = 6;
constexpr int B2_STAGE_BYTES = 128 * BLOCK_K * 2;  // this CTA's 128-row half of the 256-row B tile
// Operand kinds of oz_gemm2_kernel.  A k-block is one 128-byte swizzle row either way (64 bf16 or 128 e4m3 channels), so
// the ring, the TMA boxes' byte geometry and the 32-byte descriptor step per MMA (K = 16 bf16 / K = 32 e4m3) are shared.
constexpr int OP_BF16 = 0;       // bf16 x bf16, epilogue relu(acc + bias) -> bf16
constexpr int OP_FP8_E4M3 = 1;   // e4m3 x e4m3, epilogue relu(fma(acc, alpha, bias)) -> e4m3 (conv3, conv4; DESIGN 13)
constexpr int OP_FP8_BF16 = 2;   // e4m3 x e4m3, epilogue relu(fma(acc, alpha, bias)) -> bf16 (fc1)
template <int OP>
struct Gemm2Smem {
    static constexpr int OFF_A = 0;
    static constexpr int OFF_B = STAGES2 * A_STAGE_BYTES;
    static constexpr int OFF_BAR = OFF_B + STAGES2 * B2_STAGE_BYTES;  // full[S], empty[S], tfull[2], tempty[2]
    static constexpr int OFF_TMEM = OFF_BAR + (2 * STAGES2 + 4) * 8;
    static constexpr int OFF_BIAS = OFF_TMEM + 16;                    // [2][256] bias (+ [2][256] alpha for FP8)
    static constexpr int BYTES = OFF_BIAS + (OP == OP_BF16 ? 1 : 2) * 2 * 256 * 4;
    static constexpr int DYN_BYTES = BYTES + 1024;
};

template <int OP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
oz_gemm2_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapA2,
                const __grid_constant__ CUtensorMap mapB, const GemmParams p) {
    using S = Gemm2Smem<OP>;
    constexpr int BLOCK_N = 256;
    constexpr int KB = OP == OP_BF16 ? BLOCK_K : 2 * BLOCK_K;  // channels (tensor-map elements) per k-block
    constexpr uint32_t TMEM_COLS = 2 * BLOCK_N;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gbase = smem_raw + (base - raw);
    const uint32_t sA = base + S::OFF_A, sB = base + S::OFF_B, sBar = base + S::OFF_BAR;
    auto full_bar = [&](int s) { return sBar + 8u * s; };
    auto empty_bar = [&](int s) { return sBar + 8u * (STAGES2 + s); };
    auto tfull_bar = [&](int a) { return sBar + 8u * (2 * STAGES2 + a); };
    auto tempty_bar = [&](int a) { return sBar + 8u * (2 * STAGES2 + 2 + a); };
    volatile uint32_t* s_tmem = (volatile uint32_t*)(gbase + S::OFF_TMEM);
    float* s_bias = (float*)(gbase + S::OFF_BIAS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();  // 0 = leader (issues the MMAs)
    const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
    trace_begin(p.trace);
    int L = *p.count;
    if (L > p.max_count) L = p.max_count;
    const int m_tiles = (L * p.tile_num + p.tile_den - 1) / p.tile_den;
    const int num_pair_tiles = ((m_tiles + 1) >> 1) * p.n_tiles;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapB);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES2; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 8); }  // 4 epilogue warps x 2 CTAs
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) {
        tmem_alloc_2sm(smem_u32((const void*)s_tmem), TMEM_COLS);
        tmem_relinquish_2sm();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // both CTAs' barriers are initialised before any remote arrive / multicast commit
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    pdl_launch_dependents();

    if (warp == 0) {
        {  // ===== TMA producer (both CTAs; transaction bytes land on the LEADER's full barrier); elected lane issues =====
            pdl_wait();
            // division-free k loop, tile-invariant work hoisted: see the producer of oz_gemm_kernel
            int stage = 0; uint32_t phase = 0;
            const int ntaps_y = p.num_kb / (p.chunks_per_tap * p.ntaps_x);
            const uint32_t tx_bytes = 2u * (p.a_bytes + (unsigned)B2_STAGE_BYTES);
            const uint32_t off_main_after_half = (uint32_t)(p.half_rows * 128);
            const uint32_t off_half_after_main = (uint32_t)(p.nb * p.rows_per_board * 128);
            const uint32_t fb0 = mapa_cluster(full_bar(0), 0);  // the leader's full[0]; full[s] is 8*s bytes further
            for (int pt = cluster_id; pt < num_pair_tiles; pt += num_clusters) {
                const int m_pair = pt / p.n_tiles, n_idx = pt - m_pair * p.n_tiles;
                const int m_tile = 2 * m_pair + (int)rank;
                const int n0 = n_idx * BLOCK_N + (int)rank * 128;
                const int hb0 = m_tile * p.halves;
                const bool odd = p.split && (hb0 & 1);
                const int bA = p.split ? ((hb0 >> 1) + (odd ? 1 : 0)) : m_tile * p.nb;
                const int bH = (hb0 >> 1) + (odd ? 0 : p.nb);
                const uint32_t offA = odd ? off_main_after_half : 0u;
                const uint32_t offH = odd ? 0u : off_half_after_main;
                const int yH = odd ? p.half_h : 0;
                int kcol = 0;
                for (int ky = -p.pad; ky < ntaps_y - p.pad; ++ky) {
                    for (int kx = -p.pad; kx < p.ntaps_x - p.pad; ++kx) {
                        for (int c0 = 0; c0 < p.chunks_per_tap * KB; c0 += KB) {
                            mbar_wait(empty_bar(stage), phase ^ 1u);
                            if (elect_one()) {
                                const uint32_t fb = fb0 + 8u * (uint32_t)stage;
                                if (rank == 0) mbar_expect_tx(full_bar(stage), tx_bytes);
                                const uint32_t dstA = sA + stage * A_STAGE_BYTES;
                                tma_load_4d_2sm(dstA + offA, &mapA, fb, c0, kx, ky, bA);
                                if (p.split) tma_load_4d_2sm(dstA + offH, &mapA2, fb, c0, kx, ky + yH, bH);
                                tma_load_2d_2sm(sB + stage * B2_STAGE_BYTES, &mapB, fb, kcol, n0);
                            }
                            __syncwarp();
                            kcol += KB;
                            if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (rank == 0) {  // ===== MMA issuer: one elected lane of the leader CTA's warp drives both tensor cores =====
            constexpr uint32_t idesc = OP == OP_BF16 ? make_idesc(256, BLOCK_N) : make_idesc_e4m3(256, BLOCK_N);
            const uint32_t a_lo0 = sw128_desc_lo(sA), b_lo0 = sw128_desc_lo(sB);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int pt = cluster_id; pt < num_pair_tiles; pt += num_clusters) {
                mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BLOCK_N);
                for (int kb = 0; kb < p.num_kb; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t a_lo = a_lo0 + (uint32_t)stage * (A_STAGE_BYTES >> 4);
                    const uint32_t b_lo = b_lo0 + (uint32_t)stage * (B2_STAGE_BYTES >> 4);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {  // 4 x 32 bytes: K = 16 bf16 or 32 e4m3 per MMA
                            if constexpr (OP == OP_BF16)
                                umma_bf16_2sm_lo(d_tmem, a_lo + 2u * k, b_lo + 2u * k, idesc, (kb | k) ? 1u : 0u);
                            else
                                umma_e4m3_2sm_lo(d_tmem, a_lo + 2u * k, b_lo + 2u * k, idesc, (kb | k) ? 1u : 0u);
                        }
                        umma_commit_2sm(empty_bar(stage), 3);  // frees the stage in BOTH CTAs
                    }
                    __syncwarp();
                    if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
                }
                if (elect_one()) umma_commit_2sm(tfull_bar(acc), 3);  // accumulator complete -> both epilogues
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        const int ew = warp - 4;
        const int et = threadIdx.x - 128;
        int acc = 0; uint32_t acc_phase = 0;
        for (int pt = cluster_id; pt < num_pair_tiles; pt += num_clusters) {
            const int m_pair = pt / p.n_tiles, n_idx = pt - m_pair * p.n_tiles;
            const int m_tile = 2 * m_pair + (int)rank;
            float* bias = s_bias + acc * BLOCK_N;
            float* alpha = s_bias + (2 + acc) * BLOCK_N;  // FP8 only
            for (int i = et; i < BLOCK_N; i += 128) bias[i] = p.bias[n_idx * BLOCK_N + i];
            if constexpr (OP != OP_BF16)
                for (int i = et; i < BLOCK_N; i += 128) alpha[i] = p.alpha[n_idx * BLOCK_N + i];
            epi_bar_sync();
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
            const int r = ew * 32 + lane;
            const long long grow = (long long)m_tile * p.rows_valid + r;
            const bool ok = (r < p.rows_valid) && (grow < (long long)L * p.rows_per_board);
            const uint32_t t_row = tmem_base + (uint32_t)(acc * BLOCK_N) + ((uint32_t)(ew * 32) << 16);
            bf16* orow = p.out + grow * p.ldc + (long long)n_idx * BLOCK_N;
#pragma unroll 1
            for (int c = 0; c < BLOCK_N / 32; ++c) {
                uint32_t v[32];
                tmem_ld32(t_row + (uint32_t)(c * 32), v);
                tmem_ld_wait();
                if (ok) {
                    if constexpr (OP == OP_BF16) {
                        uint32_t packed[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float2 bj = *reinterpret_cast<const float2*>(bias + c * 32 + 2 * j);
                            const float2 y = __fadd2_rn(make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), bj);
                            packed[j] = pack_relu_bf16x2(y.x, y.y);
                        }
                        uint4* dst = reinterpret_cast<uint4*>(orow + c * 32);
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            dst[q] = make_uint4(packed[4 * q], packed[4 * q + 1], packed[4 * q + 2], packed[4 * q + 3]);
                    } else {
                        float y[32];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float2 aj = *reinterpret_cast<const float2*>(alpha + c * 32 + 2 * j);
                            const float2 bj = *reinterpret_cast<const float2*>(bias + c * 32 + 2 * j);
                            const float2 t = __ffma2_rn(make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), aj, bj);
                            y[2 * j] = t.x; y[2 * j + 1] = t.y;
                        }
                        if constexpr (OP == OP_FP8_E4M3) {  // row stride p.ldc BYTES
                            uint32_t packed[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) packed[j] = pack_relu_e4m3x4(y[4 * j], y[4 * j + 1], y[4 * j + 2], y[4 * j + 3]);
                            uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.out) + grow * p.ldc +
                                                                  (long long)n_idx * BLOCK_N + c * 32);
                            dst[0] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
                            dst[1] = make_uint4(packed[4], packed[5], packed[6], packed[7]);
                        } else {
                            uint4* dst = reinterpret_cast<uint4*>(orow + c * 32);
#pragma unroll
                            for (int q = 0; q < 4; ++q)
                                dst[q] = make_uint4(pack_relu_bf16x2(y[8 * q], y[8 * q + 1]), pack_relu_bf16x2(y[8 * q + 2], y[8 * q + 3]),
                                                    pack_relu_bf16x2(y[8 * q + 4], y[8 * q + 5]), pack_relu_bf16x2(y[8 * q + 6], y[8 * q + 7]));
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa_cluster(tempty_bar(acc), 0));  // the LEADER's barrier gates the next MMA
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // nobody exits (or frees TMEM) while the peer may still multicast into it
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    }
    trace_end(p.trace);
}

// ---- fc2 + heads in ONE kernel (opt-in, OZ_NET_TAIL=fused; a measured negative result, DESIGN 3d) --------------------------
// fc2 (4 GFLOP) and the heads (0.5 GFLOP) run as two launches of the generic kernels: 20 + 25 us per 3800 boards for 3 us of
// tensor work.  This kernel lets one CTA own 128 batch rows end to end:
//   fc2    f2[128 x 512] = relu(f1[128 x 1024] . W4'^T + b4')   two N = 256 halves, 16 k-blocks each, accumulators in TMEM
//                                                               columns [0,256) and [256,512)
//   drain  each half goes TMEM -> +bias, ReLU, bf16 -> SHARED MEMORY in the K-major 128-byte-swizzled layout tcgen05.mma
//          reads its A operand from (and to global f2, kept for inspection)
//   heads  logits[128 x 128] = f2 . W5^T: A = the f2 tile just written, B = the head weights streamed through the same TMA
//          ring; 4 k-blocks per f2 half, accumulated in TMEM columns [0,128) (free again once half 0 is drained)
//   epilogue = the heads epilogue of oz_gemm_kernel (softmax, tanh, evaluation-cache publish)
// Bit-identical to the two launches (tests/test_gpu_net.py::test_fused_tail_matches_split_launches), but NOT faster: with 128-row
// tiles only 32 CTAs exist at 4096 boards, each pulling 48 KB per k-block through a 3-deep ring (8 us per half against 4 us of
// MMA time), the drains cost 5 us each and the one-thread-per-row heads epilogue 7 us: 30 us after fc1 ends against 24 us for the
// two launches (whose prologues hide under their predecessors thanks to PDL).  The per-phase %globaltimer stamps (p.dbg) are
// what established this.
constexpr int TSTAGES = 3;
constexpr int T_B_STAGE_BYTES = 256 * BLOCK_K * 2;  // fc2: 256 weight rows per k-block; the heads use the first 16 KB
struct TailSmem {
    static constexpr int OFF_A = 0;
    static constexpr int OFF_B = TSTAGES * A_STAGE_BYTES;
    static constexpr int OFF_F2 = OFF_B + TSTAGES * T_B_STAGE_BYTES;  // one f2 half: 4 k-blocks x [128 rows x 128 B]
    static constexpr int OFF_BAR = OFF_F2 + 4 * A_STAGE_BYTES;         // full[S], empty[S], tfull[3], f2ready[2], hdone, tfree
    static constexpr int OFF_TMEM = OFF_BAR + (2 * TSTAGES + 7) * 8 + 8;
    static constexpr int OFF_BIAS = OFF_TMEM + 16;                     // [512] fc2 + [128] heads
    static constexpr int BYTES = OFF_BIAS + 640 * 4;
    static constexpr int DYN_BYTES = BYTES + 1024;
};
struct TailParams {
    int max_count;
    const int* count;
    const float* bias4; const float* bias5;
    bf16* f2;                              // [B][512], written for inspection (oz_net_get_activation)
    float* pi; float* logits; float* v;
    int nsq;
    const int* cache_idx; float* cache_pi; float* cache_v; unsigned long long* cache_tags;  // see GemmParams
    unsigned long long* trace;
    unsigned long long* dbg;  // OZ_NET_TRACE: 8 %globaltimer stamps of CTA 0 (pdl wait over, tfull0, f2ready0, tfull1, f2ready1, tfull2, logits read, done)
};

__global__ void __launch_bounds__(GEMM_THREADS, 1)
oz_tail_kernel(const __grid_constant__ CUtensorMap mapA /* f1: (1024, 1, 1, B), box (64, 1, 1, 128) */,
               const __grid_constant__ CUtensorMap mapB4 /* W4': (1024, 512), box (64, 256) */,
               const __grid_constant__ CUtensorMap mapB5 /* W5: (512, 128), box (64, 128) */, const TailParams p) {
    using S = TailSmem;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gbase = smem_raw + (base - raw);
    const uint32_t sA = base + S::OFF_A, sB = base + S::OFF_B, sF2 = base + S::OFF_F2, sBar = base + S::OFF_BAR;
    auto full_bar = [&](int s) { return sBar + 8u * s; };
    auto empty_bar = [&](int s) { return sBar + 8u * (TSTAGES + s); };
    auto tfull_bar = [&](int a) { return sBar + 8u * (2 * TSTAGES + a); };        // fc2 half 0, half 1, heads
    auto f2ready_bar = [&](int h) { return sBar + 8u * (2 * TSTAGES + 3 + h); };  // f2 half h is in shared memory
    const uint32_t hdone_bar = sBar + 8u * (2 * TSTAGES + 5);                      // heads MMAs over half 0 retired
    const uint32_t tfree_bar = sBar + 8u * (2 * TSTAGES + 6);                      // heads accumulator read out
    volatile uint32_t* s_tmem = (volatile uint32_t*)(gbase + S::OFF_TMEM);
    float* s_bias = (float*)(gbase + S::OFF_BIAS);
    uint8_t* f2buf = gbase + S::OFF_F2;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    trace_begin(p.trace);
    int L = *p.count;
    if (L > p.max_count) L = p.max_count;
    const int num_tiles = (L + BLOCK_M - 1) / BLOCK_M;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapB4);
        tma_prefetch_desc(&mapB5);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < TSTAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int a = 0; a < 3; ++a) mbar_init(tfull_bar(a), 1);
        mbar_init(f2ready_bar(0), 4); mbar_init(f2ready_bar(1), 4);  // one arrive per epilogue warp
        mbar_init(hdone_bar, 1);
        mbar_init(tfree_bar, 4);
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) {
        tmem_alloc(smem_u32((const void*)s_tmem), 512);
        tmem_relinquish();
    }
    if (warp >= 4) {  // weights, not activations: may be read before the previous layer has finished
        const int et = threadIdx.x - 128;
        for (int i = et; i < 512; i += 128) s_bias[i] = p.bias4[i];
        s_bias[512 + et] = p.bias5[et];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    pdl_launch_dependents();

    if (warp == 0) {
        // ===== TMA producer: 2 x 16 stages of (f1 k-block, 256 fc2 weight rows), then 8 stages of head weights =====
        pdl_wait();  // f1 is the previous kernel's output
        if (p.dbg && blockIdx.x == 0 && lane == 0) p.dbg[0] = global_ns();
        int stage = 0; uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int row0 = tile * BLOCK_M;
            for (int h = 0; h < 2; ++h) {
                for (int kc = 0; kc < 1024; kc += BLOCK_K) {
                    mbar_wait(empty_bar(stage), phase ^ 1u);
                    if (elect_one()) {
                        const uint32_t fb = full_bar(stage);
                        mbar_expect_tx(fb, (uint32_t)(A_STAGE_BYTES + T_B_STAGE_BYTES));
                        tma_load_4d(sA + stage * A_STAGE_BYTES, &mapA, fb, kc, 0, 0, row0);
                        tma_load_2d(sB + stage * T_B_STAGE_BYTES, &mapB4, fb, kc, h * 256);
                    }
                    __syncwarp();
                    if (++stage == TSTAGES) { stage = 0; phase ^= 1u; }
                }
            }
            for (int kc = 0; kc < 512; kc += BLOCK_K) {
                mbar_wait(empty_bar(stage), phase ^ 1u);
                if (elect_one()) {
                    const uint32_t fb = full_bar(stage);
                    mbar_expect_tx(fb, (uint32_t)A_STAGE_BYTES);  // 128 rows x 64 k of W5
                    tma_load_2d(sB + stage * T_B_STAGE_BYTES, &mapB5, fb, kc, 0);
                }
                __syncwarp();
                if (++stage == TSTAGES) { stage = 0; phase ^= 1u; }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===== MMA issuer (converged warp, elected lane) =====
        constexpr uint32_t idesc_fc2 = make_idesc(BLOCK_M, 256);
        constexpr uint32_t idesc_heads = make_idesc(BLOCK_M, 128);
        const uint32_t a_lo0 = sw128_desc_lo(sA), b_lo0 = sw128_desc_lo(sB), f_lo0 = sw128_desc_lo(sF2);
        int stage = 0; uint32_t phase = 0;
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it ^= 1u) {
            mbar_wait(tfree_bar, it ^ 1u);  // the previous tile's logits have left TMEM columns [0,128)
            tc_fence_after();
            for (int h = 0; h < 2; ++h) {
                const uint32_t d_tmem = tmem_base + (uint32_t)(h * 256);
                for (int kb = 0; kb < 16; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t a_lo = a_lo0 + (uint32_t)stage * (A_STAGE_BYTES >> 4);
                    const uint32_t b_lo = b_lo0 + (uint32_t)stage * (T_B_STAGE_BYTES >> 4);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                            umma_bf16_lo(d_tmem, a_lo + 2u * k, b_lo + 2u * k, idesc_fc2, (kb | k) ? 1u : 0u);
                        umma_commit(empty_bar(stage));
                    }
                    __syncwarp();
                    if (++stage == TSTAGES) { stage = 0; phase ^= 1u; }
                }
                if (elect_one()) umma_commit(tfull_bar(h));
                __syncwarp();
            }
            for (int h = 0; h < 2; ++h) {
                mbar_wait(f2ready_bar(h), it);  // f2 half h sits in shared memory (and, h = 0: columns [0,256) are drained)
                tc_fence_after();
                for (int kb = 0; kb < 4; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t a_lo = f_lo0 + (uint32_t)kb * (A_STAGE_BYTES >> 4);
                    const uint32_t b_lo = b_lo0 + (uint32_t)stage * (T_B_STAGE_BYTES >> 4);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                            umma_bf16_lo(tmem_base, a_lo + 2u * k, b_lo + 2u * k, idesc_heads, (h | kb | k) ? 1u : 0u);
                        umma_commit(empty_bar(stage));
                    }
                    __syncwarp();
                    if (++stage == TSTAGES) { stage = 0; phase ^= 1u; }
                }
                if (elect_one()) umma_commit(h == 0 ? hdone_bar : tfull_bar(2));
                __syncwarp();
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ===== epilogue warps: drain fc2 halves into the heads' A operand, then the heads epilogue =====
        const int ew = warp - 4;
        const int r = ew * 32 + lane;
        const uint32_t t_lane = tmem_base + ((uint32_t)(ew * 32) << 16);
        uint8_t* f2row = f2buf + (r >> 3) * 1024 + (r & 7) * 128;
        const uint32_t sw = (uint32_t)(r & 7);
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it ^= 1u) {
            const long long grow = (long long)tile * BLOCK_M + r;
            const bool ok = grow < (long long)L;
            for (int h = 0; h < 2; ++h) {
                mbar_wait(tfull_bar(h), it);
                if (p.dbg && blockIdx.x == 0 && threadIdx.x == 128) p.dbg[1 + 2 * h] = global_ns();
                if (h == 1) mbar_wait(hdone_bar, it);  // the heads MMAs have finished reading half 0 out of the buffer
                tc_fence_after();
                const float* bias = s_bias + h * 256;
                bf16* grow_out = p.f2 + grow * 512 + h * 256;
#pragma unroll 1
                for (int c = 0; c < 8; ++c) {
                    uint32_t v[32];
                    tmem_ld32(t_lane + (uint32_t)(h * 256 + c * 32), v);
                    tmem_ld_wait();
                    uint32_t packed[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float2 bj = *reinterpret_cast<const float2*>(bias + c * 32 + 2 * j);
                        const float2 y = __fadd2_rn(make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), bj);
                        packed[j] = pack_relu_bf16x2(y.x, y.y);
                    }
                    // columns c*32 .. c*32+31 of this half = k-block c/2, 16-byte chunks (c&1)*4 .. +3 of the 128-byte row,
                    // stored where the 128B swizzle (chunk ^ (row & 7)) puts them
                    uint8_t* kb_row = f2row + (c >> 1) * A_STAGE_BYTES;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const uint4 val = make_uint4(packed[4 * q], packed[4 * q + 1], packed[4 * q + 2], packed[4 * q + 3]);
                        const uint32_t ch = (uint32_t)((c & 1) * 4 + q);
                        *reinterpret_cast<uint4*>(kb_row + ((ch ^ sw) << 4)) = val;
                        if (ok) *reinterpret_cast<uint4*>(grow_out + c * 32 + q * 8) = val;
                    }
                }
                fence_proxy_async();  // generic-proxy stores -> visible to the tensor core's reads
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(f2ready_bar(h));
                if (p.dbg && blockIdx.x == 0 && threadIdx.x == 128) p.dbg[2 + 2 * h] = global_ns();
            }
            // heads: columns [0,nsq) = policy logits, column nsq = value pre-activation (same code as oz_gemm_kernel<128, EPI_HEADS>)
            mbar_wait(tfull_bar(2), it);
            if (p.dbg && blockIdx.x == 0 && threadIdx.x == 128) p.dbg[5] = global_ns();
            tc_fence_after();
            const float* bias = s_bias + 512;
            float lg[96];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                uint32_t v[32];
                tmem_ld32(t_lane + (uint32_t)(c * 32), v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j) lg[c * 32 + j] = __uint_as_float(v[j]) + bias[c * 32 + j];
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tfree_bar);  // the logits are in registers: the next tile may overwrite the accumulator
            if (p.dbg && blockIdx.x == 0 && threadIdx.x == 128) p.dbg[6] = global_ns();
            if (ok) {
                const int nsq = p.nsq;
                float mx = -3.0e38f;
#pragma unroll
                for (int j = 0; j < 64; ++j) if (j < nsq) mx = fmaxf(mx, lg[j]);
                float sum = 0.f;
                float ex[64];
#pragma unroll
                for (int j = 0; j < 64; ++j) { ex[j] = (j < nsq) ? expf(lg[j] - mx) : 0.f; sum += ex[j]; }
                const float inv = 1.0f / sum;
                float* prow = p.pi + grow * 64;
#pragma unroll
                for (int j = 0; j < 64; j += 4)
                    *reinterpret_cast<float4*>(prow + j) = make_float4(ex[j] * inv, ex[j + 1] * inv, ex[j + 2] * inv, ex[j + 3] * inv);
                if (p.logits) {
                    float* lrow = p.logits + grow * 64;
#pragma unroll
                    for (int j = 0; j < 64; j += 4)
                        *reinterpret_cast<float4*>(lrow + j) = make_float4(lg[j], lg[j + 1], lg[j + 2], lg[j + 3]);
                }
                const float val = tanhf(nsq == 64 ? lg[64] : lg[36]);
                p.v[grow] = val;
                if (p.cache_idx) {
                    const int cidx = p.cache_idx[grow];
                    if (cidx >= 0) {
                        float* crow = p.cache_pi + (size_t)cidx * 64;
#pragma unroll
                        for (int j = 0; j < 64; j += 4)
                            *reinterpret_cast<float4*>(crow + j) = make_float4(ex[j] * inv, ex[j + 1] * inv, ex[j + 2] * inv, ex[j + 3] * inv);
                        p.cache_v[cidx] = val;
                        atomicOr(p.cache_tags + cidx, 1ull);  // no fence needed: see oz_gemm_kernel's heads epilogue
                    }
                }
            }
            if (p.dbg && blockIdx.x == 0 && threadIdx.x == 128) p.dbg[7] = global_ns();
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
    trace_end(p.trace);
}

// ---- conv3 as a 1-D Winograd F(2,3) along y, on SM pairs -------------------------------------------------------------
// A 'valid' 3x3 convolution produces output rows (2ty, 2ty+1) from input rows d0..d3 = 2ty..2ty+3.  With
//     V0 = d0-d2, V1 = d1+d2, V2 = d2-d1, V3 = d1-d3               (input transform: done by the table gather, bf16)
//     U0 = g0, U1 = (g0+g1+g2)/2, U2 = (g0-g1+g2)/2, U3 = g2         (filter transform over ky: done at weight load)
//     M_e[b,ty,x][co] = sum_{kx,ci} V_e[b,ty,x+kx][ci] * U_e[co][kx,ci]            (4 GEMMs with K = 3C instead of one with 9C)
//     out[2ty] = M0 + M1 + M2,  out[2ty+1] = M1 - M2 - M3
// the layer needs 2/3 of the tensor-core work of the direct form (4 x 3 instead of 2 x 9 channel contractions per output
// pair).  M0..M3 of a tile must meet in one epilogue, so the four accumulators (128 fp32 columns each) fill the 512 TMEM
// columns of the SM; the MMA/epilogue overlap that double buffering gave the direct kernel is recovered differently: the
// epilogue first copies M0 into registers and releases accumulator 0, so the next tile's e=0 MMAs (a quarter of its main
// loop) run while this tile's outputs are combined and stored.  Rows of an M tile are (board, ty, x): 18 per 8x8 board,
// 7 boards = 126 of 128 rows.  Same SM-pair scheme as oz_gemm2_kernel (each CTA stages its 128 A rows and its 64-row half
// of the 128-row B tile: 24 KB per k-block, 8-deep ring).
constexpr int WSTAGES = 8;
constexpr int WINO_N = 128;
constexpr int WB_STAGE_BYTES = (WINO_N / 2) * BLOCK_K * 2;
constexpr int WINO_THREADS = 384;  // warp 0 TMA, 1 MMA, 2 TMEM alloc, 4..11 epilogue (two column halves per TMEM lane quarter)
struct WinoSmem {
    static constexpr int OFF_A = 0;
    static constexpr int OFF_B = WSTAGES * A_STAGE_BYTES;
    static constexpr int OFF_BAR = OFF_B + WSTAGES * WB_STAGE_BYTES;  // full[S], empty[S], tfull, tempty0, tempty123
    static constexpr int OFF_TMEM = OFF_BAR + (2 * WSTAGES + 4) * 8;
    static constexpr int OFF_BIAS = OFF_TMEM + 16;                    // [2][WINO_N] floats
    static constexpr int BYTES = OFF_BIAS + 2 * WINO_N * 4;
    static constexpr int DYN_BYTES = BYTES + 1024;
};
struct WinoParams {
    int num_kb_eta;      // 3 * C / 64: k-blocks of one transformed GEMM
    int chunks_per_tap;  // C / 64
    int nb;              // boards per M tile
    int rows_per_board;  // T * OW
    int rows_valid;      // nb * rows_per_board
    int OW, OH;          // output width / height (n-2)
    int n_tiles;         // C / 128
    int C;
    int bmax;            // boards per eta slab of V
    int max_count;
    unsigned a_bytes;
    const int* count;
    const float* bias;
    bf16* out;           // act3 [B][OH][OW][C]
    unsigned long long* trace;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(WINO_THREADS, 1)
oz_wino_kernel(const __grid_constant__ CUtensorMap mapV, const __grid_constant__ CUtensorMap mapU, const WinoParams p) {
    using S = WinoSmem;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gbase = smem_raw + (base - raw);
    const uint32_t sA = base + S::OFF_A, sB = base + S::OFF_B, sBar = base + S::OFF_BAR;
    auto full_bar = [&](int s) { return sBar + 8u * s; };
    auto empty_bar = [&](int s) { return sBar + 8u * (WSTAGES + s); };
    const uint32_t tfull_bar = sBar + 8u * (2 * WSTAGES);
    const uint32_t tempty0_bar = sBar + 8u * (2 * WSTAGES + 1);   // accumulator 0 has been copied out
    const uint32_t tempty1_bar = sBar + 8u * (2 * WSTAGES + 2);   // accumulators 1..3 have been drained
    volatile uint32_t* s_tmem = (volatile uint32_t*)(gbase + S::OFF_TMEM);
    float* s_bias = (float*)(gbase + S::OFF_BIAS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
    trace_begin(p.trace);
    int L = *p.count;
    if (L > p.max_count) L = p.max_count;
    const int m_tiles = (L + p.nb - 1) / p.nb;
    const int num_pair_tiles = ((m_tiles + 1) >> 1) * p.n_tiles;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapV);
        tma_prefetch_desc(&mapU);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < WSTAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        mbar_init(tfull_bar, 1);
        mbar_init(tempty0_bar, 16);  // 8 epilogue warps x 2 CTAs
        mbar_init(tempty1_bar, 16);
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) {
        tmem_alloc_2sm(smem_u32((const void*)s_tmem), 512);
        tmem_relinquish_2sm();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    pdl_launch_dependents();

    if (warp == 0) {
        {  // ===== TMA producer (both CTAs; bytes land on the leader's full barrier); elected lane issues =====
            pdl_wait();
            int stage = 0; uint32_t phase = 0;
            for (int pt = cluster_id; pt < num_pair_tiles; pt += num_clusters) {
                const int m_pair = pt / p.n_tiles, n_idx = pt - m_pair * p.n_tiles;
                const int m_tile = 2 * m_pair + (int)rank;
                const uint32_t tx_bytes = 2u * (p.a_bytes + (unsigned)WB_STAGE_BYTES);
                const uint32_t fb0 = mapa_cluster(full_bar(0), 0);
                for (int eta = 0; eta < 4; ++eta) {  // division-free k loop: see the producer of oz_gemm_kernel
                    const int brow = eta * p.bmax + m_tile * p.nb;
                    const int urow = eta * p.C + n_idx * WINO_N + (int)rank * (WINO_N / 2);
                    int kcol = 0;
                    for (int kx = 0; kx < 3; ++kx) {
                        for (int c0 = 0; c0 < p.chunks_per_tap * BLOCK_K; c0 += BLOCK_K) {
                            mbar_wait(empty_bar(stage), phase ^ 1u);
                            if (elect_one()) {
                                const uint32_t fb = fb0 + 8u * (uint32_t)stage;
                                if (rank == 0) mbar_expect_tx(full_bar(stage), tx_bytes);
                                tma_load_4d_2sm(sA + stage * A_STAGE_BYTES, &mapV, fb, c0, kx, 0, brow);
                                tma_load_2d_2sm(sB + stage * WB_STAGE_BYTES, &mapU, fb, kcol, urow);
                            }
                            __syncwarp();
                            kcol += BLOCK_K;
                            if (++stage == WSTAGES) { stage = 0; phase ^= 1u; }
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (rank == 0) {  // ===== MMA issuer (leader CTA) =====
            // The whole warp walks the loop (so the compiler keeps descriptors and barrier addresses in uniform registers)
            // and lane 0 issues: an N=128 instruction occupies the tensor pipe for only ~64 clk, so the issue path has to
            // stay well under that per MMA.
            constexpr uint32_t idesc = make_idesc(256, WINO_N);
            const uint32_t a_lo0 = sw128_desc_lo(sA), b_lo0 = sw128_desc_lo(sB);
            int stage = 0; uint32_t phase = 0;
            uint32_t tile_phase = 0;
            for (int pt = cluster_id; pt < num_pair_tiles; pt += num_clusters) {
                for (int eta = 0; eta < 4; ++eta) {
                    if (eta == 0) { mbar_wait(tempty0_bar, tile_phase ^ 1u); tc_fence_after(); }
                    if (eta == 1) { mbar_wait(tempty1_bar, tile_phase ^ 1u); tc_fence_after(); }
                    const uint32_t d_tmem = tmem_base + (uint32_t)(eta * WINO_N);
                    for (int kb = 0; kb < p.num_kb_eta; ++kb) {
                        mbar_wait(full_bar(stage), phase);
                        tc_fence_after();
                        const uint32_t a_lo = a_lo0 + (uint32_t)stage * (A_STAGE_BYTES >> 4);
                        const uint32_t b_lo = b_lo0 + (uint32_t)stage * (WB_STAGE_BYTES >> 4);
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                                umma_bf16_2sm_lo(d_tmem, a_lo + 2u * k, b_lo + 2u * k, idesc, (kb | k) ? 1u : 0u);
                            umma_commit_2sm(empty_bar(stage), 3);
                        }
                        __syncwarp();
                        if (++stage == WSTAGES) { stage = 0; phase ^= 1u; }
                    }
                }
                if (elect_one()) umma_commit_2sm(tfull_bar, 3);  // all four accumulators complete -> both epilogues
                __syncwarp();
                tile_phase ^= 1u;
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ===== epilogue: out[2ty] = M0+M1+M2, out[2ty+1] = M1-M2-M3 (+bias, ReLU, bf16) =====
        const int ew = warp & 3;          // TMEM lane quarter this warp may access
        const int half = (warp - 4) >> 2;  // which 64 of the 128 columns
        const int et = threadIdx.x - 128;
        uint32_t tile_phase = 0;
        int buf = 0;
        for (int pt = cluster_id; pt < num_pair_tiles; pt += num_clusters) {
            const int m_pair = pt / p.n_tiles, n_idx = pt - m_pair * p.n_tiles;
            const int m_tile = 2 * m_pair + (int)rank;
            float* bias = s_bias + buf * WINO_N;
            if (et < WINO_N) bias[et] = p.bias[n_idx * WINO_N + et];
            asm volatile("bar.sync 1, 256;" ::: "memory");
            const int r = ew * 32 + lane;
            const int bl = r / p.rows_per_board, rem = r - bl * p.rows_per_board;
            const int ty = rem / p.OW, xo = rem - ty * p.OW;
            const int b = m_tile * p.nb + bl;
            const bool ok = (r < p.rows_valid) && (b < L);
            bf16* out0 = p.out + (((long long)b * p.OH + 2 * ty) * p.OW + xo) * p.C + n_idx * WINO_N + half * 64;
            bf16* out1 = out0 + (long long)p.OW * p.C;
            const uint32_t t_row = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(half * 64);
            mbar_wait(tfull_bar, tile_phase);
            tc_fence_after();
            uint32_t m0a[32], m0b[32];
            tmem_ld32(t_row, m0a);
            tmem_ld32(t_row + 32u, m0b);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa_cluster(tempty0_bar, 0));  // the next tile's e=0 MMAs may start
            const float* bh = bias + half * 64;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                uint32_t m1[16], m2[16], m3[16];
                tmem_ld16(t_row + (uint32_t)(1 * WINO_N + c * 16), m1);
                tmem_ld16(t_row + (uint32_t)(2 * WINO_N + c * 16), m2);
                tmem_ld16(t_row + (uint32_t)(3 * WINO_N + c * 16), m3);
                tmem_ld_wait();
                uint32_t pk0[8], pk1[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float y0[2], y1[2];
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int col = c * 16 + 2 * j + h;
                        const float a0 = __uint_as_float(col < 32 ? m0a[col & 31] : m0b[col & 31]);
                        const float a1 = __uint_as_float(m1[2 * j + h]), a2 = __uint_as_float(m2[2 * j + h]);
                        const float a3 = __uint_as_float(m3[2 * j + h]);
                        const float bb = bh[col];
                        y0[h] = fmaxf(__fadd_rn(__fadd_rn(__fadd_rn(a0, a1), a2), bb), 0.0f);
                        y1[h] = fmaxf(__fadd_rn(__fsub_rn(__fsub_rn(a1, a2), a3), bb), 0.0f);
                    }
                    __nv_bfloat162 h0 = __floats2bfloat162_rn(y0[0], y0[1]);
                    __nv_bfloat162 h1 = __floats2bfloat162_rn(y1[0], y1[1]);
                    pk0[j] = *reinterpret_cast<uint32_t*>(&h0);
                    pk1[j] = *reinterpret_cast<uint32_t*>(&h1);
                }
                if (ok) {
                    uint4* d0 = reinterpret_cast<uint4*>(out0 + c * 16);
                    uint4* d1 = reinterpret_cast<uint4*>(out1 + c * 16);
                    d0[0] = make_uint4(pk0[0], pk0[1], pk0[2], pk0[3]);
                    d0[1] = make_uint4(pk0[4], pk0[5], pk0[6], pk0[7]);
                    d1[0] = make_uint4(pk1[0], pk1[1], pk1[2], pk1[3]);
                    d1[1] = make_uint4(pk1[4], pk1[5], pk1[6], pk1[7]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa_cluster(tempty1_bar, 0));
            tile_phase ^= 1u;
            buf ^= 1;
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, 512);
    }
    trace_end(p.trace);
}

// U[e][co][kx*C + ci] = bf16 of the F(2,3) filter transform over ky of the BN-folded conv kernel (Keras HWIO W[(ky*3+kx)*C+ci][co])
__global__ void wino_weights_kernel(const float* __restrict__ W, const float* __restrict__ gamma, const float* __restrict__ var,
                                    float eps, int C, bf16* __restrict__ U) {
    const size_t per_eta = (size_t)C * 3 * C, total = 4 * per_eta;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int eta = (int)(i / per_eta);
        const size_t r = i - (size_t)eta * per_eta;
        const int co = (int)(r / (3 * C)), k = (int)(r - (size_t)co * 3 * C);
        const int kx = k / C, ci = k - kx * C;
        const float s = gamma[co] / sqrtf(var[co] + eps);
        const float g0 = W[((size_t)(0 * 3 + kx) * C + ci) * C + co] * s;
        const float g1 = W[((size_t)(1 * 3 + kx) * C + ci) * C + co] * s;
        const float g2 = W[((size_t)(2 * 3 + kx) * C + ci) * C + co] * s;
        float u;
        if (eta == 0) u = g0;
        else if (eta == 1) u = __fmul_rn(__fadd_rn(__fadd_rn(g0, g1), g2), 0.5f);
        else if (eta == 2) u = __fmul_rn(__fadd_rn(__fsub_rn(g0, g1), g2), 0.5f);
        else u = g2;
        U[i] = __float2bfloat16(u);
    }
}

// ---- conv1 as a table gather -------------------------------------------------------------------------
// table[pattern][co] = relu(b' + sum_t [s_t==own] W'[t][0][co] + [s_t==opp] W'[t][1][co]), pattern = sum s_t 3^t,
// t = ky*3+kx (cross-correlation, Keras Conv2D), s = 0 empty / outside the board (zero padding), 1 own, 2 opp.
__global__ void conv1_table_kernel(const float* __restrict__ w1 /*[9][2][C]*/, const float* __restrict__ b1,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   const float* __restrict__ mean, const float* __restrict__ var, float eps, int C,
                                   bf16* __restrict__ table) {
    int pat = blockIdx.x;
    int digits[9];
    int x = pat;
    for (int t = 0; t < 9; ++t) { digits[t] = x % 3; x /= 3; }
    for (int co = threadIdx.x; co < C; co += blockDim.x) {
        float s = gamma[co] / sqrtf(var[co] + eps);
        float acc = 0.f;
        for (int t = 0; t < 9; ++t)
            if (digits[t]) acc += w1[(t * 2 + (digits[t] - 1)) * C + co];
        float y = (acc + b1[co] - mean[co]) * s + beta[co];
        table[(size_t)pat * C + co] = __float2bfloat16(fmaxf(y, 0.f));
    }
}

__global__ void __launch_bounds__(256)
conv1_gather_kernel(const u64* __restrict__ own, const u64* __restrict__ opp, const int* __restrict__ count, int max_count,
                    int n, int C, const bf16* __restrict__ table, bf16* __restrict__ out) {
    // one CTA per board: 64 threads classify the 3x3 neighbourhoods, then all 256 stream table rows -> act1
    __shared__ int s_pat[64];
    int L = *count;
    if (L > max_count) L = max_count;
    const int nsq = n * n;
    for (int b = blockIdx.x; b < L; b += gridDim.x) {
        const u64 o = own[b], q = opp[b];
        if (threadIdx.x < nsq) {
            const int pos = threadIdx.x;
            const int y = pos / n, x = pos - y * n;
            int pat = 0, mul = 1;
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
                int s = 0;
                if (yy >= 0 && yy < n && xx >= 0 && xx < n) {
                    const int bit = yy * 8 + xx;
                    s = (int)((o >> bit) & 1ull) + 2 * (int)((q >> bit) & 1ull);
                }
                pat += s * mul;
                mul *= 3;
            }
            s_pat[pos] = pat;
        }
        __syncthreads();
        const int cpr = C / 8;                 // 16-byte chunks per row
        const int total = nsq * cpr;
        uint4* dst = reinterpret_cast<uint4*>(out + (size_t)b * nsq * C);
        const uint4* tab = reinterpret_cast<const uint4*>(table);
#pragma unroll 4
        for (int i = threadIdx.x; i < total; i += 256) {
            const int pos = i / cpr, within = i - pos * cpr;
            dst[i] = __ldg(tab + (size_t)s_pat[pos] * cpr + within);
        }
        __syncthreads();
    }
}

// ---- conv1∘conv2 as a table gather ------------------------------------------------------------------------
// conv2's input at square q is table1[pat(q)], one of 3^9 vectors, so tap t's contribution W2'[t] · act1[q] to the
// output at q - offset(t) is one of 19683 x 9 pre-computable vectors:
//     table2[pat][t][co] = bf16( sum_ci W2'[co][t*C+ci] * table1[pat][ci] )      (fp32 accumulate, built at weight load
//                                                                                  by the tcgen05 GEMM below)
//     act2[b][y][x][co]  = bf16( relu( bias2'[co] + sum_{t : (y+ky-1, x+kx-1) on the board} table2[pat(y+ky-1,x+kx-1)][t][co] ) )
// i.e. 302 MFLOP per 8x8 board become <= 576 (484 on-board) 1-KB row reads + fp32 adds: the layer moves from the
// tensor roofline to the HBM/L2 roofline (484 KB read + 64 KB written per board at C=512) and conv1's output is never
// materialised.  Squares outside the board are conv2's zero padding (NOT pattern 0): they read the all-zero row
// N_PATTERNS, which stays in L1.
__global__ void permute_conv2_weights_kernel(const bf16* __restrict__ w /*[co][t*C+ci]*/, int C, bf16* __restrict__ wr /*[t*C+co][ci]*/) {
    const size_t total = 9ull * C * C;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int ci = (int)(i % C);
        const size_t r = i / C;
        const int co = (int)(r % C), t = (int)(r / C);
        wr[i] = w[(size_t)co * 9 * C + (size_t)t * C + ci];
    }
}

// One warp per output square: NJ x 9 independent 16-byte loads per lane (the whole 1-KB row of every tap), fp32x2
// accumulation.  Measured alternatives (B200, 4096 boards, C=512): half-row warp items at 62 registers / 32 warps per SM
// are SLOWER (0.28 vs 0.19 ms: the per-item address arithmetic doubles); masking the odd element instead of the fused
// pair encoding costs 20 % more instructions for the same time (the kernel is latency-, not issue-bound at 62 % issue).
// EXACT: C == 256 * NJ, i.e. every lane owns NJ full chunks: the chunk guard (a predicated load plus two register-zeroing
// instructions per load) disappears and the row stride is a compile-time constant.  s_pat holds 9 * pattern (the row
// index of tap 0).
// acc + (low 16 bits of w read as bf16), in fp32 (sm_100 mixed-precision add: one FHADD.BF16, no unpacking)
__device__ __forceinline__ float add_f32_bf16lo(float acc, uint32_t w) {
    asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %1;\n\tadd.rn.f32.bf16 %0, lo, %0;\n\t}" : "+f"(acc) : "r"(w));
    return acc;
}
constexpr int OUT_BF16 = 0;  // conv2_table_gather_kernel output kinds: act2 as bf16
constexpr int OUT_E4M3 = 1;  // act2 as e4m3 in units of its FP8 scale (DESIGN 13): 8 bytes per 16-byte table chunk
template <int NJ, bool EXACT, int OUT>
__device__ __forceinline__ void t2_square(const uint4* __restrict__ tab, const int* s_pat, int np2, int y, int x, int cpr_rt,
                                          int lane, const float2 (&bs)[NJ][4], uint4 (&res)[NJ], float out_scale) {
    const int cpr = EXACT ? 32 * NJ : cpr_rt;
    uint4 v[9][NJ];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        const int row9 = s_pat[(y + t / 3) * np2 + (x + t % 3)];  // padded coordinates of (y+ky-1, x+kx-1)
        const uint4* row = tab + (size_t)(unsigned)((row9 + t) * cpr);
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int ch = lane + 32 * j;
            v[t][j] = (EXACT || ch < cpr) ? __ldg(row + ch) : make_uint4(0, 0, 0, 0);
        }
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        // 6 instructions per 16-byte chunk: the even (low-half) elements are added with the mixed-precision
        // add.f32.bf16 (FHADD.BF16 reads the register half directly - no shift), the odd ones two words at a time with
        // add.f32x2 on the words themselves (see pack_pair_fused).  Same roundings as shift + fp32 add.
        float ev[4];
        float2 od[2];
#pragma unroll
        for (int i = 0; i < 4; ++i) ev[i] = bs[j][i].x;
        od[0] = make_float2(bs[j][0].y, bs[j][1].y);
        od[1] = make_float2(bs[j][2].y, bs[j][3].y);
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const uint32_t w4[4] = {v[t][j].x, v[t][j].y, v[t][j].z, v[t][j].w};
#pragma unroll
            for (int i = 0; i < 4; ++i) ev[i] = add_f32_bf16lo(ev[i], w4[i]);
            od[0] = __fadd2_rn(od[0], make_float2(__uint_as_float(w4[0]), __uint_as_float(w4[1])));
            od[1] = __fadd2_rn(od[1], make_float2(__uint_as_float(w4[2]), __uint_as_float(w4[3])));
        }
        if constexpr (OUT == OUT_BF16)
            res[j] = make_uint4(pack_relu_bf16x2(ev[0], od[0].x), pack_relu_bf16x2(ev[1], od[0].y),
                                pack_relu_bf16x2(ev[2], od[1].x), pack_relu_bf16x2(ev[3], od[1].y));
        else  // channels 0..7 of the chunk are ev0, od0.x, ev1, od0.y, ev2, od1.x, ev3, od1.y
            res[j] = make_uint4(pack_relu_e4m3x4(ev[0] * out_scale, od[0].x * out_scale, ev[1] * out_scale, od[0].y * out_scale),
                                pack_relu_e4m3x4(ev[2] * out_scale, od[1].x * out_scale, ev[3] * out_scale, od[1].y * out_scale), 0u, 0u);
    }
}

__device__ __forceinline__ uint32_t bf2_add(uint32_t a, uint32_t b) {
    __nv_bfloat162 r = __hadd2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t bf2_sub(uint32_t a, uint32_t b) {
    __nv_bfloat162 r = __hsub2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint4 bf8_add(const uint4& a, const uint4& b) {
    return make_uint4(bf2_add(a.x, b.x), bf2_add(a.y, b.y), bf2_add(a.z, b.z), bf2_add(a.w, b.w));
}
__device__ __forceinline__ uint4 bf8_sub(const uint4& a, const uint4& b) {
    return make_uint4(bf2_sub(a.x, b.x), bf2_sub(a.y, b.y), bf2_sub(a.z, b.z), bf2_sub(a.w, b.w));
}

// WINO = false: writes act2 [B][n][n][C].
// WINO = true : conv3 runs as the Winograd kernel above, so act2 itself is never stored; a warp walks one board column
//               top to bottom, keeps the previous two (bf16-rounded) squares in registers and stores the input transform
//               V [4][Bmax][T][n][C]:  V0 = d0-d2, V1 = d1+d2, V2 = d2-d1 when row 2ty+2 arrives, V3 = d1-d3 at row 2ty+3
//               (bf16 subtraction of bf16 values: one rounding of the exact difference).
// OUT = OUT_E4M3 (FP8 networks, WINO = false): act2 [B][n][n][C] as e4m3 bytes, e4m3_rn(relu(acc) * bias[C]); `bias` then
//               holds C biases followed by 1 / sa_2, the reciprocal of act2's FP8 scale.
template <int NJ, bool WINO, bool EXACT, int OUT>  // 16-byte chunks per lane: C <= 256 * NJ (C = 128: NJ = 1, upper half-warp idle)
__global__ void __launch_bounds__(256, 2)
conv2_table_gather_kernel(const u64* __restrict__ own, const u64* __restrict__ opp, const int* __restrict__ count,
                          int max_count, int n, int C, const bf16* __restrict__ table2, const float* __restrict__ bias,
                          bf16* __restrict__ out, int bmax, unsigned long long* trace) {
    __shared__ int s_pat[100];  // (n+2) x (n+2) patterns with a border of N_PATTERNS (the zero row)
    trace_begin(trace);
    int L = *count;
    if (L > max_count) L = max_count;
    const int nsq = n * n, np2 = n + 2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cpr = EXACT ? 32 * NJ : (C >> 3);  // 16-byte chunks per row
    float2 bs[NJ][4];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int ch = lane + 32 * j;
#pragma unroll
        for (int i = 0; i < 4; ++i)
            bs[j][i] = (EXACT || ch < cpr) ? make_float2(bias[ch * 8 + 2 * i], bias[ch * 8 + 2 * i + 1]) : make_float2(0.f, 0.f);
    }
    const uint4* tab = reinterpret_cast<const uint4*>(table2);
    const float out_scale = OUT == OUT_E4M3 ? bias[C] : 1.0f;
    for (int b = blockIdx.x; b < L; b += gridDim.x) {
        const u64 o = own[b], q = opp[b];
        if (threadIdx.x < np2 * np2) {
            const int py = threadIdx.x / np2, px = threadIdx.x - py * np2;
            const int y = py - 1, x = px - 1;
            int pat = N_PATTERNS;  // stored as 9 * pattern = row index of tap 0 in table2
            if (y >= 0 && y < n && x >= 0 && x < n) {
                pat = 0;
                int mul = 1;
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                    const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
                    int s = 0;
                    if (yy >= 0 && yy < n && xx >= 0 && xx < n) {
                        const int bit = yy * 8 + xx;
                        s = (int)((o >> bit) & 1ull) + 2 * (int)((q >> bit) & 1ull);
                    }
                    pat += s * mul;
                    mul *= 3;
                }
            }
            s_pat[threadIdx.x] = pat * 9;
        }
        __syncthreads();
        if constexpr (!WINO) {
            for (int pos = warp; pos < nsq; pos += 8) {
                const int y = pos / n, x = pos - y * n;
                uint4 res[NJ];
                t2_square<NJ, EXACT, OUT>(tab, s_pat, np2, y, x, cpr, lane, bs, res, out_scale);
                if constexpr (OUT == OUT_BF16) {
                    uint4* orow = reinterpret_cast<uint4*>(out + ((size_t)b * nsq + pos) * C);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const int ch = lane + 32 * j;
                        if (EXACT || ch < cpr) orow[ch] = res[j];
                    }
                } else {
                    uint2* orow = reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(out) + ((size_t)b * nsq + pos) * C);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const int ch = lane + 32 * j;
                        if (EXACT || ch < cpr) orow[ch] = make_uint2(res[j].x, res[j].y);
                    }
                }
            }
        } else {
            const int T = (n - 2) >> 1;
            const size_t eta_stride = (size_t)bmax * T * n * cpr;  // uint4 units
            uint4* vout = reinterpret_cast<uint4*>(out);
            for (int x = warp; x < n; x += 8) {
                uint4 p2[NJ] = {}, p1[NJ] = {};
#pragma unroll 1
                for (int y = 0; y < n; ++y) {
                    uint4 cur[NJ];
                    t2_square<NJ, EXACT, OUT>(tab, s_pat, np2, y, x, cpr, lane, bs, cur, out_scale);
                    if (y >= 2) {
                        if (!(y & 1)) {
                            const int ty = (y - 2) >> 1;
                            uint4* v0 = vout + (((size_t)b * T + ty) * n + x) * cpr;
#pragma unroll
                            for (int j = 0; j < NJ; ++j) {
                                const int ch = lane + 32 * j;
                                if (EXACT || ch < cpr) {
                                    v0[ch] = bf8_sub(p2[j], cur[j]);
                                    v0[eta_stride + ch] = bf8_add(p1[j], cur[j]);
                                    v0[2 * eta_stride + ch] = bf8_sub(cur[j], p1[j]);
                                }
                            }
                        } else {
                            const int ty = (y - 3) >> 1;
                            uint4* v3 = vout + 3 * eta_stride + (((size_t)b * T + ty) * n + x) * cpr;
#pragma unroll
                            for (int j = 0; j < NJ; ++j) {
                                const int ch = lane + 32 * j;
                                if (EXACT || ch < cpr) v3[ch] = bf8_sub(p2[j], cur[j]);
                            }
                        }
                    }
#pragma unroll
                    for (int j = 0; j < NJ; ++j) { p2[j] = p1[j]; p1[j] = cur[j]; }
                }
            }
        }
        __syncthreads();
    }
    trace_end(trace);
}

// ---- weight folding -------------------------------------------------------------------------------------
// Keras kernel W[k][o] (HWIO flattened / Dense (in,out)) -> Wt[o][k] bf16 with the BN scale folded;
// bias'[o] = (b - mean) * s + beta.
__global__ void fold_weights_kernel(const float* __restrict__ W, const float* __restrict__ b, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, const float* __restrict__ mean,
                                    const float* __restrict__ var, float eps, int K, int Nout, bf16* __restrict__ Wt,
                                    float* __restrict__ bias_out) {
    __shared__ float tile[32][33];
    const int k0 = blockIdx.x * 32, o0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int k = k0 + i, o = o0 + threadIdx.x;
        tile[i][threadIdx.x] = (k < K && o < Nout) ? W[(size_t)k * Nout + o] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int o = o0 + i, k = k0 + threadIdx.x;
        if (o < Nout && k < K) {
            float s = gamma ? gamma[o] / sqrtf(var[o] + eps) : 1.0f;
            Wt[(size_t)o * K + k] = __float2bfloat16(tile[threadIdx.x][i] * s);
        }
    }
    if (blockIdx.x == 0 && threadIdx.y == 0) {
        int o = o0 + threadIdx.x;
        if (o < Nout) {
            float s = gamma ? gamma[o] / sqrtf(var[o] + eps) : 1.0f;
            bias_out[o] = gamma ? (b[o] - mean[o]) * s + beta[o] : b[o];
        }
    }
}

// ---- FP8 evaluation (DESIGN 13): load-time quantisation and calibration -------------------------------------------------
// Wq[o][k] = e4m3_rn_satfinite(W'[k][o] / sw[o]) with W' the BN-folded fp32 weight (the same product fold_weights_kernel
// casts to bf16) and sw[o] = amax_k |W'[k][o]| / 448 (1 for an all-zero channel).  A block owns 32 output channels.
__global__ void quantize_weights_e4m3_kernel(const float* __restrict__ W, const float* __restrict__ gamma,
                                             const float* __restrict__ var, float eps, int K, int Nout,
                                             uint8_t* __restrict__ Wq, float* __restrict__ sw) {
    __shared__ float red[8][33];
    const int o = blockIdx.x * 32 + threadIdx.x;
    const bool on = o < Nout;
    const float s = on ? gamma[o] / sqrtf(var[o] + eps) : 0.f;
    float m = 0.f;
    if (on)
        for (int k = threadIdx.y; k < K; k += blockDim.y) m = fmaxf(m, fabsf(W[(size_t)k * Nout + o] * s));
    red[threadIdx.y][threadIdx.x] = m;
    __syncthreads();
    for (int i = 0; i < 8; ++i) m = fmaxf(m, red[i][threadIdx.x]);
    const float scale = m > 0.f ? m / 448.0f : 1.0f;
    if (!on) return;
    if (threadIdx.y == 0) sw[o] = scale;
    for (int k = threadIdx.y; k < K; k += blockDim.y)
        Wq[(size_t)o * K + k] = (uint8_t)__nv_cvt_float_to_fp8(W[(size_t)k * Nout + o] * s / scale, __NV_SATFINITE, __NV_E4M3);
}

// Largest value of the first count*per_board elements of a (non-negative, post-ReLU) bf16 activation, folded into *out
// as fp32 bits (non-negative floats order like their bit patterns).
__global__ void amax_bf16_kernel(const int* __restrict__ count, int max_count, const bf16* __restrict__ x, long long per_board,
                                 unsigned* __restrict__ out) {
    int L = *count;
    if (L > max_count) L = max_count;
    const long long n = (long long)L * per_board;
    float m = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = fmaxf(m, __bfloat162float(x[i]));
    const unsigned u = __reduce_max_sync(0xffffffffu, __float_as_uint(m));
    if ((threadIdx.x & 31) == 0 && u) atomicMax(out, u);
}

// Epilogue coefficients of an FP8 layer: alpha[o] = sa_in * sw[o] / sa_out, beta[o] = bias[o] / sa_out.
__global__ void fp8_coef_kernel(const float* __restrict__ sw, const float* __restrict__ bias, float sa_in, float sa_out, int n,
                                float* __restrict__ alpha, float* __restrict__ beta) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    alpha[i] = sa_in * sw[i] / sa_out;
    beta[i] = bias[i] / sa_out;
}

typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_tmapEncodeTiled get_encode_fn() {
    static PFN_tmapEncodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_tmapEncodeTiled)p;
    }
    return fn;
}

}  // namespace

struct OzLayer {
    CUtensorMap mapA, mapA2, mapB, mapB2;
    bool use_2sm = false;
    GemmParams p;
    int block_n;
    int epi;
    int op = OP_BF16;  // operand kind of the SM-pair kernel (FP8 layers: OP_FP8_*)
    int max_tiles;
    double flops_per_board;
};

// Calibration set of the FP8 activation scales (DESIGN 13): every position (side to move's frame) of CAL_GAMES uniformly
// random games under the reference rules, from the RNG streams stream_key(CAL_SEED, game).
constexpr int CAL_GAMES = 256;
constexpr u64 CAL_SEED = 0xCA11B7A7Eull;

struct OzNet {
    int n = 0, C = 0, Bmax = 0;
    bool loaded = false;
    bool timing = false;
    bool pdl = true;
    int timing_every = 16;   // per-layer events on every 16th forward only (an event between two kernels breaks their PDL edge)
    long forwards = 0;
    int sm_count = 148;
    bf16* table1 = nullptr;
    // conv1∘conv2 partial-product table [19683 + 1 zero row][9 taps][C] (OZ_NET_CONV2=gemm keeps the implicit GEMM instead)
    bool conv2_table = true;
    bf16* table2 = nullptr; bf16* w2perm = nullptr; float* zero_bias = nullptr; int* d_npat = nullptr;
    OzLayer tbl;
    // conv3 as 1-D Winograd F(2,3): OZ_NET_CONV3=wino (needs conv2_table: the gather emits the input transform)
    bool conv3_wino = false;
    bool fused_tail = false;  // OZ_NET_TAIL=fused: fc2 + heads as oz_tail_kernel (a measured negative result, DESIGN 3d)
    bf16* v3 = nullptr;      // [4][Bmax][T][n][C]
    bf16* u3 = nullptr;      // [4][C][3C]
    CUtensorMap mapV, mapU;
    WinoParams wp;
    unsigned long long* trace = nullptr;  // OZ_NET_TRACE: [trace_slots][2]
    int trace_slots = 0, trace_next = 0;
    char trace_name[256][12];
    bf16 *w[6] = {nullptr}; float* bias[6] = {nullptr};  // conv2, conv3, conv4, fc1, fc2, heads
    bf16 *act1 = nullptr, *act2 = nullptr, *act3 = nullptr, *act4 = nullptr, *f1 = nullptr, *f2 = nullptr;
    OzLayer layer[6];
    // FP8 evaluation (OZ_NET_FP8, fixed at the first load): conv3, conv4, fc1 as layer8[0..2].  The bf16 layers stay
    // set up: the calibration forward runs the bf16 gather, conv3 and conv4.
    bool fp8 = false;
    uint8_t* w8[3] = {nullptr};                       // [Nout][K] e4m3
    float *sw8[3] = {nullptr}, *alpha8[3] = {nullptr}, *beta8[3] = {nullptr};
    float* gcoef = nullptr;                           // the FP8 gather's bias[C] + 1 / sa_2
    uint8_t *act2_8 = nullptr, *act3_8 = nullptr, *act4_8 = nullptr;
    OzLayer layer8[3];
    float sa[3] = {1.f, 1.f, 1.f};                   // act2, act3, act4
    u64 *cal_own = nullptr, *cal_opp = nullptr;
    int* cal_counts = nullptr;                        // boards of each Bmax-sized chunk
    int cal_positions = 0;
    unsigned* d_amax = nullptr;
    // per-layer timing: a ring of event sets, harvested lazily so the stream is never blocked
    static constexpr int RING = 8;
    cudaEvent_t ev[RING][8] = {{nullptr}};
    bool ev_used[RING] = {false};
    int ev_next = 0;
    double ms_sum[8] = {0};
    long ms_cnt = 0;
    void* allocs[64];
    int n_allocs = 0;
};

static void oz_net_harvest(OzNet* net, int r) {
    cudaEventSynchronize(net->ev[r][7]);  // RING forwards old when called from the hot loop: already complete
    for (int i = 0; i < 7; ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, net->ev[r][i], net->ev[r][i + 1]) == cudaSuccess) net->ms_sum[i] += ms;
    }
    net->ms_cnt++;
    net->ev_used[r] = false;
}

static int net_alloc(OzNet* net, void** p, size_t bytes) {
    cudaError_t err = cudaMalloc(p, bytes + 256);
    if (err != cudaSuccess) { oz_set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(err)); return OZ_ERR_NOMEM; }
    net->allocs[net->n_allocs++] = *p;
    return OZ_OK;
}

int64_t oz_net_blob_floats_impl(int n, int C) {
    if ((n != 6 && n != 8) || C <= 0) return -1;
    int64_t nsq = n * n, k1 = (int64_t)(n - 4) * (n - 4) * C;
    int64_t t = 0;
    t += 18LL * C + C + 4LL * C;                 // conv1 + bn1
    t += 3 * (9LL * C * C + C + 4LL * C);        // conv2..4 + bn
    t += k1 * 1024 + 1024 + 4 * 1024;            // fc1 + bn5
    t += 1024LL * 512 + 512 + 4 * 512;           // fc2 + bn6
    t += 512 * nsq + nsq;                        // pi
    t += 512 + 1;                                // v
    return t;
}

int oz_net_create(oz_engine* e) {
    e->net = nullptr;
    if (e->cfg.prior_mode != OZ_PRIOR_NET) return OZ_OK;
    OzNet* net = new OzNet();
    net->n = e->cfg.board_size;
    net->Bmax = e->cfg.max_games * (e->cfg.vl_width > 1 ? e->cfg.vl_width : 1);
    const char* t = getenv("OZ_NET_TIMING");
    net->timing = t && t[0] == '1';
    const char* pd = getenv("OZ_NET_NO_PDL");
    net->pdl = !(pd && pd[0] == '1');
    const char* c2 = getenv("OZ_NET_CONV2");
    net->conv2_table = !(c2 && c2[0] == 'g');
    const char* c3 = getenv("OZ_NET_CONV3");
    net->conv3_wino = net->conv2_table && c3 && c3[0] == 'w';  // opt-in: measured at parity with the direct kernel (DESIGN 3b)
    const char* tl = getenv("OZ_NET_TAIL");
    net->fused_tail = tl && tl[0] == 'f';  // opt-in: measured slower than the two generic launches (DESIGN 3d)
    const char* tr = getenv("OZ_NET_TRACE");
    if (tr && atoi(tr) > 0) net->trace_slots = atoi(tr) > 256 ? 256 : atoi(tr);
    const char* te = getenv("OZ_NET_TIMING_EVERY");
    if (te && atoi(te) > 0) net->timing_every = atoi(te);
    int dev = e->cfg.device;
    cudaDeviceGetAttribute(&net->sm_count, cudaDevAttrMultiProcessorCount, dev);
    for (int r = 0; r < OzNet::RING; ++r)
        for (int i = 0; i < 8; ++i) cudaEventCreate(&net->ev[r][i]);
    e->net = net;
    return OZ_OK;
}

static unsigned long long* trace_slot(OzNet* net, const char* name) {
    if (!net->trace || net->trace_next >= net->trace_slots) return nullptr;
    snprintf(net->trace_name[net->trace_next], sizeof(net->trace_name[0]), "%s", name);
    return net->trace + 2 * (net->trace_next++);
}

static void trace_dump(OzNet* net) {
    if (!net->trace || net->trace_next == 0) return;
    cudaDeviceSynchronize();
    unsigned long long* h = (unsigned long long*)malloc(sizeof(unsigned long long) * 2 * net->trace_next);
    cudaMemcpy(h, net->trace, sizeof(unsigned long long) * 2 * net->trace_next, cudaMemcpyDeviceToHost);
    unsigned long long t0 = ~0ull;
    for (int i = 0; i < net->trace_next; ++i) if (h[2 * i] < t0) t0 = h[2 * i];
    for (int i = 0; i < net->trace_next; ++i)
        fprintf(stderr, "OZ_TRACE %3d %-8s start %9.1f us  end %9.1f us  dur %8.1f us\n", i, net->trace_name[i],
                (h[2 * i] - t0) / 1e3, (h[2 * i + 1] - t0) / 1e3, (h[2 * i + 1] - h[2 * i]) / 1e3);
    free(h);
}

void oz_net_destroy(oz_engine* e) {
    OzNet* net = e->net;
    if (!net) return;
    trace_dump(net);
    for (int i = 0; i < net->n_allocs; ++i) cudaFree(net->allocs[i]);
    for (int r = 0; r < OzNet::RING; ++r)
        for (int i = 0; i < 8; ++i) if (net->ev[r][i]) cudaEventDestroy(net->ev[r][i]);
    delete net;
    e->net = nullptr;
}

// es = element bytes: 2 (bf16) or 1 (e4m3, as UINT8).  The inner box is one 128-byte swizzle row either way.
static int make_map_A(CUtensorMap* m, void* base, int Cdim, int W, int H, int B, int bw, int bh, int nb, int es = 2) {
    PFN_tmapEncodeTiled enc = get_encode_fn();
    if (!enc) { oz_set_error("cuTensorMapEncodeTiled entry point not available"); return OZ_ERR_CUDA; }
    cuuint64_t dims[4] = {(cuuint64_t)Cdim, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)Cdim * es, (cuuint64_t)Cdim * es * W, (cuuint64_t)Cdim * es * W * H};
    cuuint32_t box[4] = {(cuuint32_t)(128 / es), (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)nb};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(m, es == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, base, dims, strides, box,
                     estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { oz_set_error("cuTensorMapEncodeTiled(A) failed: %d", (int)r); return OZ_ERR_CUDA; }
    return OZ_OK;
}

static int make_map_B(CUtensorMap* m, void* base, int K, int Nout, int block_n, int es = 2) {
    PFN_tmapEncodeTiled enc = get_encode_fn();
    if (!enc) { oz_set_error("cuTensorMapEncodeTiled entry point not available"); return OZ_ERR_CUDA; }
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)Nout};
    cuuint64_t strides[1] = {(cuuint64_t)K * es};
    cuuint32_t box[2] = {(cuuint32_t)(128 / es), (cuuint32_t)block_n};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, es == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box,
                     estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { oz_set_error("cuTensorMapEncodeTiled(B) failed: %d", (int)r); return OZ_ERR_CUDA; }
    return OZ_OK;
}

static bool allow_2sm() {
    static const bool allow = !(getenv("OZ_NET_NO_2SM") && getenv("OZ_NET_NO_2SM")[0] == '1');
    return allow;
}

// layer li: input [B][ih][iw][cin] -> output [B][oh*ow][nout]; ntaps 3 (conv) or 1 (fc).  op != OP_BF16: e4m3 weights and
// input (FP8 layers, SM-pair kernel only), epilogue coefficients alpha / bias.
static int setup_layer(OzNet* net, OzLayer& Lr, void* weights, const float* bias, int bmax, void* in, int cin, int iw, int ih,
                       int ow, int oh, int ntaps, int pad, int nout_pad, int block_n, int epi, void* out, int ldc,
                       int op = OP_BF16, const float* alpha = nullptr) {
    const int es = op == OP_BF16 ? 2 : 1;  // operand element bytes
    GemmParams& p = Lr.p;
    memset(&p, 0, sizeof(p));
    if (epi == EPI_RELU_BF16) block_n = (nout_pad % 256 == 0) ? 256 : 128;
    if (epi == EPI_LINEAR_BF16) block_n = (nout_pad % 256 == 0) ? 256 : 128;
    const int rows_per_board = ow * oh;
    int nb = BLOCK_M / rows_per_board;
    if (nb > 256) nb = 256;
    p.nb = nb;
    p.rows_per_board = rows_per_board;
    p.rows_valid = nb * rows_per_board;
    p.tile_num = 1;
    p.tile_den = nb;
    static const bool allow_split = !(getenv("OZ_NET_NO_SPLIT") && getenv("OZ_NET_NO_SPLIT")[0] == '1');
    if (allow_split && ntaps == 3 && (oh % 2) == 0 && (BLOCK_M - nb * rows_per_board) * 2 >= rows_per_board) {
        p.split = 1;
        p.half_h = oh / 2;
        p.half_rows = (oh / 2) * ow;
        p.halves = 2 * nb + 1;
        p.rows_valid = p.halves * p.half_rows;
        p.tile_num = 2;
        p.tile_den = p.halves;
    }
    p.ntaps_x = ntaps;
    p.pad = pad;
    p.chunks_per_tap = cin / (128 / es);  // k-blocks of 128 bytes
    p.num_kb = ntaps * ntaps * p.chunks_per_tap;
    p.n_tiles = nout_pad / block_n;
    p.ldc = ldc;
    p.max_count = bmax;
    p.a_bytes = (unsigned)(p.rows_valid * BLOCK_K * 2);  // 128 bytes per row in either operand kind
    p.bias = bias;
    p.alpha = alpha;
    p.out = (bf16*)out;
    p.nsq = net->n * net->n;
    Lr.block_n = block_n;
    Lr.epi = epi;
    Lr.op = op;
    Lr.max_tiles = ((bmax * p.tile_num + p.tile_den - 1) / p.tile_den) * p.n_tiles;
    int rc = make_map_A(&Lr.mapA, in, cin, iw, ih, bmax, ow, oh, nb, es);
    if (rc) return rc;
    rc = make_map_A(&Lr.mapA2, in, cin, iw, ih, bmax, ow, p.split ? oh / 2 : oh, p.split ? 1 : nb, es);
    if (rc) return rc;
    // measured (B200, 4096 boards, division-free producers): the SM-pair kernel wins everywhere it applies - conv3 (split
    // tiles) 0.471 vs 0.518 ms, conv4 0.212 vs 0.231, fc1 0.062 vs 0.067: at the power cap the halved B-operand traffic
    // is clock headroom.  (With the old producer loop, which was the supply limit, the two kernels tied.)
    Lr.use_2sm = allow_2sm() && epi == EPI_RELU_BF16 && block_n == 256;
    if (op != OP_BF16 && !Lr.use_2sm) {
        oz_set_error("FP8 layers run on the SM-pair GEMM only (OZ_NET_NO_2SM=1, or an output width that is not a multiple of 256)");
        return OZ_ERR_STATE;
    }
    if (Lr.use_2sm) {
        rc = make_map_B(&Lr.mapB2, weights, ntaps * ntaps * cin, nout_pad, 128, es);
        if (rc) return rc;
    }
    return make_map_B(&Lr.mapB, weights, ntaps * ntaps * cin, nout_pad, block_n, es);
}

// One launch of the SM-pair GEMM for layer Lr (cfg carries the stream and the PDL attribute).
static cudaError_t launch_gemm2(OzNet* net, cudaLaunchConfig_t cfg, const OzLayer& Lr, const GemmParams& p, int max_count) {
    int m_tiles = (max_count * p.tile_num + p.tile_den - 1) / p.tile_den;
    int pairs = ((m_tiles + 1) / 2) * p.n_tiles;
    int g2 = 2 * pairs < (net->sm_count & ~1) ? 2 * pairs : (net->sm_count & ~1);
    if (g2 < 2) g2 = 2;
    cfg.gridDim = dim3(g2);
    switch (Lr.op) {
        case OP_FP8_E4M3:
            cfg.dynamicSmemBytes = Gemm2Smem<OP_FP8_E4M3>::DYN_BYTES;
            return cudaLaunchKernelEx(&cfg, oz_gemm2_kernel<OP_FP8_E4M3>, Lr.mapA, Lr.mapA2, Lr.mapB2, p);
        case OP_FP8_BF16:
            cfg.dynamicSmemBytes = Gemm2Smem<OP_FP8_BF16>::DYN_BYTES;
            return cudaLaunchKernelEx(&cfg, oz_gemm2_kernel<OP_FP8_BF16>, Lr.mapA, Lr.mapA2, Lr.mapB2, p);
        default:
            cfg.dynamicSmemBytes = Gemm2Smem<OP_BF16>::DYN_BYTES;
            return cudaLaunchKernelEx(&cfg, oz_gemm2_kernel<OP_BF16>, Lr.mapA, Lr.mapA2, Lr.mapB2, p);
    }
}

// 16-byte chunks per lane of conv2_table_gather_kernel for C channels: a lane covers 256 channels per chunk, so C needs
// ceil(C / 256) of them.
constexpr int gather_nj(int C) { return (C + 255) / 256; }
constexpr bool gather_nj_covers_all_channel_counts() {
    for (int C = 128; C <= 1024; C += 128)
        if (256 * gather_nj(C) < C || gather_nj(C) > 4) return false;
    return true;
}
static_assert(gather_nj_covers_all_channel_counts(), "the gather must cover every channel count oz_net_load accepts");

// conv1∘conv2 as the table gather: act2 in bf16 (out_kind OUT_BF16; or the Winograd input transform) or e4m3 (OUT_E4M3).
static void launch_gather(OzNet* net, cudaStream_t st, const u64* own_dev, const u64* opp_dev, const int* count_dev,
                          int max_count, int out_kind, unsigned long long* ts) {
    const int n = net->n, C = net->C;
    int blocks = max_count < net->sm_count * 2 ? max_count : net->sm_count * 2;  // 2 resident CTAs/SM, grid-stride
    const bf16* t2 = net->table2; const float* b2 = net->bias[0];
#define OZ_T2K(NJ, W, X, O, B, OUT) conv2_table_gather_kernel<NJ, W, X, O><<<blocks, 256, 0, st>>>(own_dev, opp_dev, count_dev, max_count, n, C, t2, B, OUT, net->Bmax, ts)
#define OZ_T2(NJ)                                                                                                       \
    if (out_kind == OUT_E4M3) OZ_T2K(NJ, false, true, OUT_E4M3, net->gcoef, (bf16*)net->act2_8);   /* C == 256 * NJ */  \
    else if (net->conv3_wino) { if (C == 256 * NJ) OZ_T2K(NJ, true, true, OUT_BF16, b2, net->v3); else OZ_T2K(NJ, true, false, OUT_BF16, b2, net->v3); } \
    else { if (C == 256 * NJ) OZ_T2K(NJ, false, true, OUT_BF16, b2, net->act2); else OZ_T2K(NJ, false, false, OUT_BF16, b2, net->act2); }
    switch (gather_nj(C)) {
        case 1: OZ_T2(1); break;
        case 2: OZ_T2(2); break;
        case 3: OZ_T2(3); break;
        default: OZ_T2(4); break;
    }
#undef OZ_T2
#undef OZ_T2K
}

// Every position of the calibration games (see CAL_GAMES), in the frame of the side to move.
static void calibration_positions(int n, std::vector<u64>& own, std::vector<u64>& opp) {
    const u64 full = ozbb::full_mask(n);
    for (int g = 0; g < CAL_GAMES; ++g) {
        const u64 key = ozbb::stream_key(CAL_SEED, (u64)g);
        u64 o, q;
        ozbb::initial_position(n, &o, &q);  // BLACK moves first
        u64 legal = ozbb::legal_moves(o, q, full);
        for (int ply = 0; legal; ++ply) {
            own.push_back(o);
            opp.push_back(q);
            const int sq = ozbb::kth_set_bit(legal, (int)ozbb::pick_index(ozbb::sm64(key + (u64)ply), (unsigned)ozbb::popc(legal)));
            ozbb::play_move<ozbb::RULES_REFERENCE>(1ull << sq, &o, &q, full, &legal);
        }
    }
}

// FP8 activation scales: the calibration set through the bf16 gather, conv3 and conv4 in chunks of Bmax boards, the
// largest act2 / act3 / act4 value over all of it.  A max is order-free and the tower is row-independent, so the result
// depends on the weights, the board size and the channel count only.
static int fp8_calibrate(oz_engine* e, OzNet* net) {
    cudaStream_t st = e->stream;
    const int n = net->n, C = net->C, B = net->Bmax;
    OZ_CUDA(cudaMemsetAsync(net->d_amax, 0, 3 * sizeof(unsigned), st));
    const long long per_board[3] = {(long long)n * n * C, (long long)(n - 2) * (n - 2) * C, (long long)(n - 4) * (n - 4) * C};
    const bf16* acts[3] = {net->act2, net->act3, net->act4};
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(GEMM_THREADS);
    cfg.stream = st;
    for (int c = 0; c * B < net->cal_positions; ++c) {
        const int cnt = net->cal_positions - c * B < B ? net->cal_positions - c * B : B;
        const int* count = net->cal_counts + c;
        launch_gather(net, st, net->cal_own + (size_t)c * B, net->cal_opp + (size_t)c * B, count, cnt, OUT_BF16, nullptr);
        OZ_CUDA(cudaGetLastError());
        for (int li = 1; li <= 2; ++li) {
            GemmParams p = net->layer[li].p;
            p.count = count;
            p.max_count = cnt;
            OZ_CUDA(launch_gemm2(net, cfg, net->layer[li], p, cnt));
        }
        for (int l = 0; l < 3; ++l) {
            long long total = cnt * per_board[l];
            int blocks = (int)((total + 255) / 256) < net->sm_count * 4 ? (int)((total + 255) / 256) : net->sm_count * 4;
            amax_bf16_kernel<<<blocks, 256, 0, st>>>(count, cnt, acts[l], per_board[l], net->d_amax + l);
        }
        OZ_CUDA(cudaGetLastError());
        e->launches += 6;
    }
    unsigned amax[3];
    OZ_CUDA(cudaMemcpyAsync(amax, net->d_amax, sizeof(amax), cudaMemcpyDeviceToHost, st));
    OZ_CUDA(cudaStreamSynchronize(st));
    for (int l = 0; l < 3; ++l) {
        float a;
        memcpy(&a, &amax[l], 4);
        net->sa[l] = a > 0.f ? a / 448.0f : 1.0f;  // an all-zero activation: any scale represents it
    }
    return OZ_OK;
}

int oz_net_load(oz_engine* e, const float* blob, int64_t n_floats, int channels, bool on_device) {
    OzNet* net = e->net;
    if (!net) { oz_set_error("engine was not created with OZ_PRIOR_NET"); return OZ_ERR_STATE; }
    const bool fp8 = (channels & OZ_NET_FP8) != 0;
    const int n = net->n, C = channels & ~OZ_NET_FP8, nsq = n * n, B = net->Bmax;
    OZ_REQUIRE(C >= 128 && C % 128 == 0 && C <= 1024, "channels must be a multiple of 128 in [128,1024] (got %d)", C);
    const int64_t need = oz_net_blob_floats_impl(n, C);
    OZ_REQUIRE(n_floats == need, "weight blob has %lld floats, expected %lld", (long long)n_floats, (long long)need);
    if (net->loaded && net->C != C) { oz_set_error("channel count cannot change after the first load"); return OZ_ERR_STATE; }
    if (net->loaded && net->fp8 != fp8) {
        oz_set_error("precision cannot change after the first load (this engine's network is %s)", net->fp8 ? "fp8" : "bf16");
        return OZ_ERR_STATE;
    }
    if (fp8) {
        OZ_REQUIRE(C % 256 == 0, "FP8 evaluation needs channels to be a multiple of 256 (got %d)", C);
        if (!net->conv2_table) { oz_set_error("FP8 evaluation needs the conv1∘conv2 table gather, but OZ_NET_CONV2=gemm is set"); return OZ_ERR_STATE; }
        if (net->conv3_wino) { oz_set_error("FP8 evaluation needs the direct conv3 kernel, but OZ_NET_CONV3=wino is set"); return OZ_ERR_STATE; }
        if (!allow_2sm()) { oz_set_error("FP8 evaluation runs on the SM-pair GEMM, but OZ_NET_NO_2SM=1 is set"); return OZ_ERR_STATE; }
    }
    cudaStream_t st = e->stream;
    const int o2 = n - 2, o4 = n - 4;
    const int K1 = o4 * o4 * C;
    int rc;
    if (!net->loaded) {
        net->C = C;
        const size_t kc = 9ull * C * C;
#define NA(ptr, bytes) if ((rc = net_alloc(net, (void**)&(ptr), (bytes)))) return rc;
        NA(net->table1, (size_t)N_PATTERNS * C * 2)
        NA(net->w[0], kc * 2) NA(net->w[1], kc * 2) NA(net->w[2], kc * 2)
        NA(net->w[3], (size_t)K1 * 1024 * 2) NA(net->w[4], 1024ull * 512 * 2) NA(net->w[5], 128ull * 512 * 2)
        NA(net->bias[0], C * 4) NA(net->bias[1], C * 4) NA(net->bias[2], C * 4)
        NA(net->bias[3], 1024 * 4) NA(net->bias[4], 512 * 4) NA(net->bias[5], 128 * 4)
        NA(net->act1, (size_t)B * nsq * C * 2)
        if (!net->conv3_wino) NA(net->act2, (size_t)B * nsq * C * 2)
        NA(net->act3, (size_t)B * o2 * o2 * C * 2) NA(net->act4, (size_t)B * o4 * o4 * C * 2)
        NA(net->f1, (size_t)B * 1024 * 2) NA(net->f2, (size_t)B * 512 * 2)
        if (net->trace_slots) {
            NA(net->trace, (size_t)net->trace_slots * 16)
            OZ_CUDA(cudaMemsetAsync(net->trace, 0, (size_t)net->trace_slots * 16, st));
            for (int i = 0; i < net->trace_slots; ++i) OZ_CUDA(cudaMemsetAsync(net->trace + 2 * i, 0xff, 8, st));
        }
        if (net->conv2_table) {
            NA(net->table2, (size_t)(N_PATTERNS + 1) * 9 * C * 2) NA(net->w2perm, kc * 2)
            NA(net->zero_bias, 9ull * C * 4) NA(net->d_npat, 16)
        }
        if (net->conv3_wino) {
            NA(net->v3, 4ull * B * ((n - 2) / 2) * n * C * 2) NA(net->u3, 4ull * C * 3 * C * 2)
            OZ_CUDA(cudaMemsetAsync(net->v3, 0, 4ull * B * ((n - 2) / 2) * n * C * 2, st));
        }
#undef NA
#define SL(li, ...) if ((rc = setup_layer(net, net->layer[li], net->w[li], net->bias[li], B, __VA_ARGS__))) return rc;
        SL(0, net->act1, C, n, n, n, n, 3, 1, C, 256, EPI_RELU_BF16, net->act2, C)
        SL(1, net->act2, C, n, n, o2, o2, 3, 0, C, 256, EPI_RELU_BF16, net->act3, C)
        SL(2, net->act3, C, o2, o2, o4, o4, 3, 0, C, 256, EPI_RELU_BF16, net->act4, C)
        SL(3, net->act4, K1, 1, 1, 1, 1, 1, 0, 1024, 256, EPI_RELU_BF16, net->f1, 1024)
        SL(4, net->f1, 1024, 1, 1, 1, 1, 1, 0, 512, 256, EPI_RELU_BF16, net->f2, 512)
        SL(5, net->f2, 512, 1, 1, 1, 1, 1, 0, 128, 128, EPI_HEADS, nullptr, 64)
#undef SL
        if (net->conv3_wino) {
            WinoParams& wp = net->wp;
            memset(&wp, 0, sizeof(wp));
            const int T = o2 / 2;
            wp.chunks_per_tap = C / BLOCK_K;
            wp.num_kb_eta = 3 * wp.chunks_per_tap;
            wp.rows_per_board = T * o2;
            wp.nb = BLOCK_M / wp.rows_per_board;
            wp.rows_valid = wp.nb * wp.rows_per_board;
            wp.OW = o2; wp.OH = o2;
            wp.n_tiles = C / WINO_N;
            wp.C = C;
            wp.bmax = B;
            wp.max_count = B;
            wp.a_bytes = (unsigned)(wp.rows_valid * BLOCK_K * 2);
            wp.bias = net->bias[1];
            wp.out = net->act3;
            // V as (C, x = n, ty = T, eta*Bmax + board): the box for tap kx is (64 channels, OW, T, nb) at x = kx
            if ((rc = make_map_A(&net->mapV, net->v3, C, n, T, 4 * B, o2, T, wp.nb))) return rc;
            if ((rc = make_map_B(&net->mapU, net->u3, 3 * C, 4 * C, WINO_N / 2))) return rc;
            OZ_CUDA(cudaFuncSetAttribute(oz_wino_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WinoSmem::DYN_BYTES));
        }
        if (net->conv2_table) {
            // table2 = table1 [19683 x C] x W2perm^T [C x 9C]: one "fc" launch of the GEMM kernel with a linear epilogue
            if ((rc = setup_layer(net, net->tbl, net->w2perm, net->zero_bias, N_PATTERNS, net->table1, C, 1, 1, 1, 1, 1, 0,
                                  9 * C, 256, EPI_LINEAR_BF16, net->table2, 9 * C))) return rc;
            OZ_CUDA(cudaFuncSetAttribute(oz_gemm_kernel<256, EPI_LINEAR_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         GemmSmem<256>::DYN_BYTES));
            OZ_CUDA(cudaFuncSetAttribute(oz_gemm_kernel<128, EPI_LINEAR_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         GemmSmem<128>::DYN_BYTES));
            OZ_CUDA(cudaFuncSetAttribute(oz_gemm_kernel<128, EPI_LINEAR_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         GemmSmem<128>::DYN_BYTES));
            OZ_CUDA(cudaMemsetAsync(net->table2 + (size_t)N_PATTERNS * 9 * C, 0, 9ull * C * 2, st));  // the padding row
            OZ_CUDA(cudaMemsetAsync(net->zero_bias, 0, 9ull * C * 4, st));
            const int npat = N_PATTERNS;
            OZ_CUDA(cudaMemcpyAsync(net->d_npat, &npat, sizeof(int), cudaMemcpyHostToDevice, st));
            OZ_CUDA(cudaStreamSynchronize(st));
        }
        OZ_CUDA(cudaFuncSetAttribute(oz_gemm_kernel<256, EPI_RELU_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     GemmSmem<256>::DYN_BYTES));
        OZ_CUDA(cudaFuncSetAttribute(oz_gemm_kernel<128, EPI_HEADS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     GemmSmem<128>::DYN_BYTES));
        OZ_CUDA(cudaFuncSetAttribute(oz_gemm_kernel<128, EPI_RELU_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     GemmSmem<128>::DYN_BYTES));
        OZ_CUDA(cudaFuncSetAttribute(oz_gemm2_kernel<OP_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     Gemm2Smem<OP_BF16>::DYN_BYTES));
        OZ_CUDA(cudaFuncSetAttribute(oz_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TailSmem::DYN_BYTES));
        OZ_CUDA(cudaMemsetAsync(net->w[5], 0, 128ull * 512 * 2, st));
        OZ_CUDA(cudaMemsetAsync(net->bias[5], 0, 128 * 4, st));
        if (fp8) {
            net->fp8 = true;
            const int kin[3] = {9 * C, 9 * C, K1}, nout[3] = {C, C, 1024};
            for (int i = 0; i < 3; ++i) {
                if ((rc = net_alloc(net, (void**)&net->w8[i], (size_t)kin[i] * nout[i]))) return rc;
                if ((rc = net_alloc(net, (void**)&net->sw8[i], (size_t)nout[i] * 4))) return rc;
                if ((rc = net_alloc(net, (void**)&net->alpha8[i], (size_t)nout[i] * 4))) return rc;
                if ((rc = net_alloc(net, (void**)&net->beta8[i], (size_t)nout[i] * 4))) return rc;
            }
            if ((rc = net_alloc(net, (void**)&net->gcoef, (size_t)(C + 1) * 4))) return rc;
            if ((rc = net_alloc(net, (void**)&net->act2_8, (size_t)B * nsq * C))) return rc;
            if ((rc = net_alloc(net, (void**)&net->act3_8, (size_t)B * o2 * o2 * C))) return rc;
            if ((rc = net_alloc(net, (void**)&net->act4_8, (size_t)B * o4 * o4 * C))) return rc;
            if ((rc = net_alloc(net, (void**)&net->d_amax, 16))) return rc;
            if ((rc = setup_layer(net, net->layer8[0], net->w8[0], net->beta8[0], B, net->act2_8, C, n, n, o2, o2, 3, 0, C, 256,
                                  EPI_RELU_BF16, net->act3_8, C, OP_FP8_E4M3, net->alpha8[0]))) return rc;
            if ((rc = setup_layer(net, net->layer8[1], net->w8[1], net->beta8[1], B, net->act3_8, C, o2, o2, o4, o4, 3, 0, C, 256,
                                  EPI_RELU_BF16, net->act4_8, C, OP_FP8_E4M3, net->alpha8[1]))) return rc;
            if ((rc = setup_layer(net, net->layer8[2], net->w8[2], net->beta8[2], B, net->act4_8, K1, 1, 1, 1, 1, 1, 0, 1024, 256,
                                  EPI_RELU_BF16, net->f1, 1024, OP_FP8_BF16, net->alpha8[2]))) return rc;
            OZ_CUDA(cudaFuncSetAttribute(oz_gemm2_kernel<OP_FP8_E4M3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Gemm2Smem<OP_FP8_E4M3>::DYN_BYTES));
            OZ_CUDA(cudaFuncSetAttribute(oz_gemm2_kernel<OP_FP8_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Gemm2Smem<OP_FP8_BF16>::DYN_BYTES));
            std::vector<u64> own, opp;
            calibration_positions(n, own, opp);
            net->cal_positions = (int)own.size();
            const int chunks = (net->cal_positions + B - 1) / B;
            std::vector<int> counts(chunks);
            for (int c = 0; c < chunks; ++c) counts[c] = net->cal_positions - c * B < B ? net->cal_positions - c * B : B;
            if ((rc = net_alloc(net, (void**)&net->cal_own, own.size() * 8))) return rc;
            if ((rc = net_alloc(net, (void**)&net->cal_opp, opp.size() * 8))) return rc;
            if ((rc = net_alloc(net, (void**)&net->cal_counts, (size_t)chunks * 4))) return rc;
            OZ_CUDA(cudaMemcpyAsync(net->cal_own, own.data(), own.size() * 8, cudaMemcpyHostToDevice, st));
            OZ_CUDA(cudaMemcpyAsync(net->cal_opp, opp.data(), opp.size() * 8, cudaMemcpyHostToDevice, st));
            OZ_CUDA(cudaMemcpyAsync(net->cal_counts, counts.data(), (size_t)chunks * 4, cudaMemcpyHostToDevice, st));
            OZ_CUDA(cudaStreamSynchronize(st));
        }
    }
    // stage the blob on the device
    const float* d = blob;
    struct Staged {  // freed on every return path (the OZ_CUDA macros return early)
        float* p = nullptr;
        cudaStream_t st;
        ~Staged() { if (p) { cudaStreamSynchronize(st); cudaFree(p); } }
    } staged;
    staged.st = st;
    if (!on_device) {
        OZ_CUDA(cudaMalloc((void**)&staged.p, (size_t)need * 4));
        OZ_CUDA(cudaMemcpyAsync(staged.p, blob, (size_t)need * 4, cudaMemcpyHostToDevice, st));
        d = staged.p;
    }
    const float eps = 1e-3f;  // keras BatchNormalization default epsilon
    const float* q = d;
    auto take = [&](int64_t cnt) { const float* r = q; q += cnt; return r; };
    dim3 tb(32, 8);
    const float *q_w[3], *q_g[3], *q_v[3];  // fp32 conv3, conv4, fc1 kernels and BN scale inputs (FP8 quantisation)
    {   // conv1 + bn1 -> table
        const float* w1 = take(18LL * C); const float* b1 = take(C);
        const float* g = take(C); const float* be = take(C); const float* mu = take(C); const float* va = take(C);
        conv1_table_kernel<<<N_PATTERNS, 256, 0, st>>>(w1, b1, g, be, mu, va, eps, C, net->table1);
        OZ_CUDA(cudaGetLastError());
        e->launches++;
    }
    for (int li = 0; li < 3; ++li) {  // conv2..4
        const int K = 9 * C;
        const float* w = take((int64_t)K * C); const float* b = take(C);
        const float* g = take(C); const float* be = take(C); const float* mu = take(C); const float* va = take(C);
        fold_weights_kernel<<<dim3((K + 31) / 32, (C + 31) / 32), tb, 0, st>>>(w, b, g, be, mu, va, eps, K, C, net->w[li], net->bias[li]);
        OZ_CUDA(cudaGetLastError());
        e->launches++;
        if (li > 0) { q_w[li - 1] = w; q_g[li - 1] = g; q_v[li - 1] = va; }
        if (li == 1 && net->conv3_wino) {
            wino_weights_kernel<<<net->sm_count * 8, 256, 0, st>>>(w, g, va, eps, C, net->u3);
            OZ_CUDA(cudaGetLastError());
            e->launches++;
        }
    }
    if (net->conv2_table) {  // table2[pat][t][:] = W2'[t] . table1[pat]  (93 GFLOP at C=512, once per weight load)
        permute_conv2_weights_kernel<<<net->sm_count * 8, 256, 0, st>>>(net->w[0], C, net->w2perm);
        OZ_CUDA(cudaGetLastError());
        OzLayer& Lr = net->tbl;
        GemmParams p = Lr.p;
        p.count = net->d_npat;
        cudaLaunchConfig_t cfg{};
        cfg.blockDim = dim3(GEMM_THREADS);
        cfg.gridDim = dim3(Lr.max_tiles < net->sm_count ? Lr.max_tiles : net->sm_count);
        cfg.stream = st;
        if (Lr.block_n == 256) {
            cfg.dynamicSmemBytes = GemmSmem<256>::DYN_BYTES;
            OZ_CUDA(cudaLaunchKernelEx(&cfg, oz_gemm_kernel<256, EPI_LINEAR_BF16>, Lr.mapA, Lr.mapA2, Lr.mapB, p));
        } else {
            cfg.dynamicSmemBytes = GemmSmem<128>::DYN_BYTES;
            OZ_CUDA(cudaLaunchKernelEx(&cfg, oz_gemm_kernel<128, EPI_LINEAR_BF16>, Lr.mapA, Lr.mapA2, Lr.mapB, p));
        }
        e->launches += 2;
    }
    {   // fc1 + bn5
        const float* w = take((int64_t)K1 * 1024); const float* b = take(1024);
        const float* g = take(1024); const float* be = take(1024); const float* mu = take(1024); const float* va = take(1024);
        fold_weights_kernel<<<dim3((K1 + 31) / 32, 32), tb, 0, st>>>(w, b, g, be, mu, va, eps, K1, 1024, net->w[3], net->bias[3]);
        OZ_CUDA(cudaGetLastError());
        e->launches++;
        q_w[2] = w; q_g[2] = g; q_v[2] = va;
    }
    {   // fc2 + bn6
        const float* w = take(1024LL * 512); const float* b = take(512);
        const float* g = take(512); const float* be = take(512); const float* mu = take(512); const float* va = take(512);
        fold_weights_kernel<<<dim3(32, 16), tb, 0, st>>>(w, b, g, be, mu, va, eps, 1024, 512, net->w[4], net->bias[4]);
        OZ_CUDA(cudaGetLastError());
        e->launches++;
    }
    {   // heads: pi rows [0,nsq), v row nsq; no BN
        const float* wp = take(512LL * nsq); const float* bp = take(nsq);
        const float* wv = take(512); const float* bv = take(1);
        fold_weights_kernel<<<dim3(16, (nsq + 31) / 32), tb, 0, st>>>(wp, bp, nullptr, nullptr, nullptr, nullptr, eps, 512, nsq,
                                                                      net->w[5], net->bias[5]);
        OZ_CUDA(cudaGetLastError());
        fold_weights_kernel<<<dim3(16, 1), tb, 0, st>>>(wv, bv, nullptr, nullptr, nullptr, nullptr, eps, 512, 1,
                                                        net->w[5] + (size_t)nsq * 512, net->bias[5] + nsq);
        OZ_CUDA(cudaGetLastError());
        e->launches += 2;
    }
    if (net->fp8) {  // DESIGN 13: quantise conv3 / conv4 / fc1, calibrate the activation scales, build the epilogue coefficients
        const int kin[3] = {9 * C, 9 * C, K1}, nout[3] = {C, C, 1024};
        for (int i = 0; i < 3; ++i) {
            quantize_weights_e4m3_kernel<<<(nout[i] + 31) / 32, tb, 0, st>>>(q_w[i], q_g[i], q_v[i], eps, kin[i], nout[i], net->w8[i],
                                                                             net->sw8[i]);
            OZ_CUDA(cudaGetLastError());
            e->launches++;
        }
        if ((rc = fp8_calibrate(e, net))) return rc;  // synchronises: the staged blob is no longer read after this
        const float sa_out[3] = {net->sa[1], net->sa[2], 1.0f};  // fc1 writes bf16 in real units
        for (int i = 0; i < 3; ++i) {
            fp8_coef_kernel<<<(nout[i] + 255) / 256, 256, 0, st>>>(net->sw8[i], net->bias[i + 1], net->sa[i], sa_out[i], nout[i],
                                                                   net->alpha8[i], net->beta8[i]);
            OZ_CUDA(cudaGetLastError());
            e->launches++;
        }
        const float inv_sa2 = 1.0f / net->sa[0];
        OZ_CUDA(cudaMemcpyAsync(net->gcoef, net->bias[0], (size_t)C * 4, cudaMemcpyDeviceToDevice, st));
        OZ_CUDA(cudaMemcpyAsync(net->gcoef + C, &inv_sa2, 4, cudaMemcpyHostToDevice, st));
    }
    OZ_CUDA(cudaStreamSynchronize(st));
    net->loaded = true;
    return OZ_OK;
}

int oz_net_scales(oz_engine* e, float* out) {
    OzNet* net = e->net;
    if (!net || !net->loaded || !net->fp8) {
        oz_set_error("no FP8 network is loaded (oz_net_load_weights with OZ_NET_FP8)");
        return OZ_ERR_STATE;
    }
    const int C = net->C;
    for (int l = 0; l < 3; ++l) out[l] = net->sa[l];
    OZ_CUDA(cudaMemcpyAsync(out + 3, net->sw8[0], (size_t)C * 4, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(out + 3 + C, net->sw8[1], (size_t)C * 4, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaMemcpyAsync(out + 3 + 2 * C, net->sw8[2], 1024 * 4, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}

int oz_net_forward(oz_engine* e, const u64* own_dev, const u64* opp_dev, const int* count_dev, int max_count,
                   float* pi_dev, float* logits_dev, float* v_dev, bool publish) {
    OzNet* net = e->net;
    if (!net || !net->loaded) { oz_set_error("network weights have not been loaded (oz_net_load_weights)"); return OZ_ERR_STATE; }
    cudaStream_t st = e->stream;
    const int n = net->n, C = net->C, nsq = n * n;
    if (max_count > net->Bmax) max_count = net->Bmax;
    const bool tm = net->timing && (net->forwards++ % net->timing_every) == 0;
    cudaEvent_t* ev = net->ev[net->ev_next];
    if (tm) {
        if (net->ev_used[net->ev_next]) oz_net_harvest(net, net->ev_next);
        net->ev_used[net->ev_next] = true;
        net->ev_next = (net->ev_next + 1) % OzNet::RING;
        cudaEventRecord(ev[0], st);
    }
    (void)nsq;
    if (!net->conv2_table) {
        int blocks = max_count < net->sm_count * 8 ? max_count : net->sm_count * 8;  // 8 resident CTAs/SM, grid-stride
        conv1_gather_kernel<<<blocks, 256, 0, st>>>(own_dev, opp_dev, count_dev, max_count, n, C, net->table1, net->act1);
        OZ_CUDA(cudaGetLastError());
        e->launches++;
    }
    if (tm) cudaEventRecord(ev[1], st);
    if (net->conv2_table) {  // conv1 + conv2 in one gather-sum over the partial-product table
        launch_gather(net, st, own_dev, opp_dev, count_dev, max_count, net->fp8 ? OUT_E4M3 : OUT_BF16, trace_slot(net, "gather"));
        OZ_CUDA(cudaGetLastError());
        e->launches++;
        if (tm) cudaEventRecord(ev[2], st);
    }
    for (int li = net->conv2_table ? 1 : 0; li < 6; ++li) {
        OzLayer& Lr = (net->fp8 && li >= 1 && li <= 3) ? net->layer8[li - 1] : net->layer[li];
        GemmParams p = Lr.p;
        p.count = count_dev;
        p.max_count = max_count;
        static const char* lname[6] = {"conv2", "conv3", "conv4", "fc1", "fc2", "heads"};
        if (li == 5 && net->fused_tail) {  // the heads ran inside the fc2 launch
            if (tm) cudaEventRecord(ev[2 + li], st);
            continue;
        }
        p.trace = (li == 4 && net->fused_tail) ? nullptr : trace_slot(net, lname[li]);
        p.pi = pi_dev; p.logits = logits_dev; p.v = v_dev;
        if (publish && li == 5) {
            p.cache_idx = e->tp.leaf_cache_idx; p.cache_pi = e->tp.cache_pi; p.cache_v = e->tp.cache_v;
            p.cache_tags = e->tp.cache_tags;
        }
        int tiles = ((max_count * p.tile_num + p.tile_den - 1) / p.tile_den) * p.n_tiles;
        int grid = tiles < net->sm_count ? tiles : net->sm_count;
        if (grid < 1) grid = 1;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cudaLaunchConfig_t cfg{};
        cfg.blockDim = dim3(GEMM_THREADS);
        cfg.stream = st;
        cfg.attrs = attr;
        cfg.numAttrs = net->pdl ? 1 : 0;
        cudaError_t lerr;
        if (li == 4 && net->fused_tail) {
            TailParams tp{};
            tp.max_count = max_count;
            tp.count = count_dev;
            tp.bias4 = net->bias[4]; tp.bias5 = net->bias[5];
            tp.f2 = net->f2;
            tp.pi = pi_dev; tp.logits = logits_dev; tp.v = v_dev;
            tp.nsq = nsq;
            if (publish) {
                tp.cache_idx = e->tp.leaf_cache_idx; tp.cache_pi = e->tp.cache_pi; tp.cache_v = e->tp.cache_v;
                tp.cache_tags = e->tp.cache_tags;
            }
            tp.trace = trace_slot(net, "fc2+heads");
            if (tp.trace && net->trace_next + 4 <= net->trace_slots) {  // 4 more slots = 8 stamps of CTA 0
                tp.dbg = trace_slot(net, "t:w,f0"); trace_slot(net, "t:r0,f1"); trace_slot(net, "t:r1,f2"); trace_slot(net, "t:lg,end");
            }
            const int m_tiles = (max_count + BLOCK_M - 1) / BLOCK_M;
            cfg.gridDim = dim3(m_tiles < net->sm_count ? (m_tiles < 1 ? 1 : m_tiles) : net->sm_count);
            cfg.dynamicSmemBytes = TailSmem::DYN_BYTES;
            lerr = cudaLaunchKernelEx(&cfg, oz_tail_kernel, Lr.mapA, Lr.mapB, net->layer[5].mapB, tp);
        } else if (li == 1 && net->conv3_wino) {
            WinoParams wp = net->wp;
            wp.count = count_dev;
            wp.max_count = max_count;
            wp.trace = p.trace;
            const int m_tiles = (max_count + wp.nb - 1) / wp.nb;
            const int pairs = ((m_tiles + 1) / 2) * wp.n_tiles;
            int g2 = 2 * pairs < (net->sm_count & ~1) ? 2 * pairs : (net->sm_count & ~1);
            if (g2 < 2) g2 = 2;
            cfg.blockDim = dim3(WINO_THREADS);
            cfg.gridDim = dim3(g2);
            cfg.dynamicSmemBytes = WinoSmem::DYN_BYTES;
            lerr = cudaLaunchKernelEx(&cfg, oz_wino_kernel, net->mapV, net->mapU, wp);
        } else if (Lr.use_2sm) {
            lerr = launch_gemm2(net, cfg, Lr, p, max_count);
        } else if (Lr.epi == EPI_RELU_BF16 && Lr.block_n == 256) {
            cfg.gridDim = dim3(grid);
            cfg.dynamicSmemBytes = GemmSmem<256>::DYN_BYTES;
            lerr = cudaLaunchKernelEx(&cfg, oz_gemm_kernel<256, EPI_RELU_BF16>, Lr.mapA, Lr.mapA2, Lr.mapB, p);
        } else if (Lr.epi == EPI_RELU_BF16) {
            cfg.gridDim = dim3(grid);
            cfg.dynamicSmemBytes = GemmSmem<128>::DYN_BYTES;
            lerr = cudaLaunchKernelEx(&cfg, oz_gemm_kernel<128, EPI_RELU_BF16>, Lr.mapA, Lr.mapA2, Lr.mapB, p);
        } else {
            cfg.gridDim = dim3(grid);
            cfg.dynamicSmemBytes = GemmSmem<128>::DYN_BYTES;
            lerr = cudaLaunchKernelEx(&cfg, oz_gemm_kernel<128, EPI_HEADS>, Lr.mapA, Lr.mapA2, Lr.mapB, p);
        }
        OZ_CUDA(lerr);
        OZ_CUDA(cudaGetLastError());
        e->launches++;
        if (tm) cudaEventRecord(ev[2 + li], st);
    }
    return OZ_OK;
}

void oz_net_set_timing_impl(oz_engine* e, bool on) {
    if (e->net) e->net->timing = on;
}

// Average per-layer device time (ms) over the forwards recorded since the last call; [7] = forwards averaged.
int oz_net_times(oz_engine* e, float* ms8) {
    OzNet* net = e->net;
    for (int i = 0; i < 8; ++i) ms8[i] = 0.f;
    if (!net) return OZ_OK;
    for (int r = 0; r < OzNet::RING; ++r)
        if (net->ev_used[r]) oz_net_harvest(net, r);
    if (net->ms_cnt > 0)
        for (int i = 0; i < 7; ++i) ms8[i] = (float)(net->ms_sum[i] / (double)net->ms_cnt);
    ms8[7] = (float)net->ms_cnt;
    for (int i = 0; i < 8; ++i) net->ms_sum[i] = 0;
    net->ms_cnt = 0;
    return OZ_OK;
}

int oz_net_activation(oz_engine* e, int layer, void* host, int64_t bytes) {
    OzNet* net = e->net;
    if (!net || !net->loaded) { oz_set_error("network not loaded"); return OZ_ERR_STATE; }
    const int n = net->n, C = net->C, B = net->Bmax;
    void* ptrs[6] = {net->act1, net->act2, net->act3, net->act4, net->f1, net->f2};
    int64_t sizes[6] = {(int64_t)B * n * n * C, (int64_t)B * n * n * C, (int64_t)B * (n - 2) * (n - 2) * C,
                        (int64_t)B * (n - 4) * (n - 4) * C, (int64_t)B * 1024, (int64_t)B * 512};
    OZ_REQUIRE(layer >= 0 && layer < 6, "layer %d out of range", layer);
    int64_t es = 2;  // element bytes
    if (net->fp8 && layer >= 1 && layer <= 3) {  // e4m3 bytes
        ptrs[layer] = layer == 1 ? net->act2_8 : layer == 2 ? net->act3_8 : net->act4_8;
        es = 1;
    }
    if (layer == 0 && net->conv2_table) {
        oz_set_error("conv1's output is not materialised while conv2 runs as the table gather (OZ_NET_CONV2=gemm keeps it)");
        return OZ_ERR_STATE;
    }
    if (layer == 1 && net->conv3_wino) {
        oz_set_error("conv2's output is not materialised while conv3 runs as the Winograd kernel (the default OZ_NET_CONV3=direct keeps it)");
        return OZ_ERR_STATE;
    }
    OZ_REQUIRE(bytes >= 0 && bytes <= sizes[layer] * es, "bytes out of range");
    OZ_CUDA(cudaMemcpyAsync(host, ptrs[layer], (size_t)bytes, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}
