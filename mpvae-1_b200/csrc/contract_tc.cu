// tcgen05 contraction engine (sm_100a): split-precision tensor-core GEMMs for the dense regime of the probit ELBO
// (label / rank sets >= 128, e.g. the delicious and eurlex shapes).
//
//   nt: nr[m, l]  = sum_z noise[m, z] * R[l, z]        both operands K-major     (mpvae.py:168)
//   tn: g_R[l, z] = sum_m gxs[m, l]  * noise[m, z]     both operands MN-major    (SURVEY 8a-12)
//
// A 10/11-bit mantissa on the operands cannot hold the 1e-5 parity bar, so every fp32 operand x is split by a
// streaming pre-pass into hi + lo, two fp16 pieces of x * s with s = 2^k chosen per tensor (common.cuh), ~22 bits
// together, and the product is accumulated in fp32 in tensor memory as  A_lo.B_hi + A_hi.B_lo + A_hi.B_hi  (the dropped
// lo.lo term is ~2^-22 relative); the result is rescaled by 1 / (s_a * s_b), exactly.
//
// The tensor core adds into its fp32 accumulator with truncation toward zero, so a long K chain drifts
// (K = 3993: -2.4e-5 relative, measured).  The accumulation is therefore chunked: tensor memory only ever holds
// `kc` k-blocks; sixteen promotion warps add each chunk into fp32 REGISTER accumulators (round-to-nearest) while
// the tensor core fills the other TMEM buffer, and scale the chunk by (1 + bias * k-blocks) to take the systematic
// part of the truncation out again (profiles/r1_tc_chunk_experiment.txt).
//
// Kernel anatomy: CTA pairs (cta_group::2), one pair per two neighbouring SMs, persistent over 256 x 256 output tiles.
//   warp 0      : TMA producer  -- cp.async.bulk.tensor (128B-swizzled boxes) into a 3- or 4-stage smem ring
//   warp 1      : MMA issuer    -- one lane of the pair's leader issues tcgen05.mma.cta_group::2 (M256 N256 K16)
//   warp 2      : TMEM allocator (512 columns = two 128 x 256 fp32 chunk accumulators per CTA, ping-pong)
//   [FUSE only] warps 4-11: row math of the probit forward on finished tiles (fused_rows.cuh)
//   last 16     : promotion + epilogue -- tcgen05.ld a chunk (32 rows x 64 columns per warp), add into registers,
//                 store the finished tile
// Pipelines: smem full/empty mbarriers (TMA <-> MMA), tmem full/empty mbarriers (MMA <-> promotion).
// The tf32 operand kind, the single-CTA kernel and the four-CTA multicast clusters of round 1 measured no gain on
// B200 (profiles/r1_tc_chunk_experiment.txt, profiles/r01_multicast_probe.txt) and were removed.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "fused_rows.cuh"
#include "philox.cuh"
#include "tc.h"

namespace mpv {
namespace {

constexpr int BM = 128, BN = 256;                        // per-CTA rows / pair columns of an output tile
constexpr int A_BYTES = BM * 128;                        // 16 KiB: BM rows x one 128-byte swizzle row (64 halves of K)
constexpr int BAR_BYTES = 256;
constexpr int TMEM_COLS = 512;
constexpr int kCtrlWarps = 4;
constexpr int kEpiWarps = 16;                            // 4 TMEM lane quadrants x 4 column quarters
constexpr int HB = BN / 2;                               // B-tile columns staged by each CTA of a pair

// MATH 1..3 add eight math warps; MATH 4 only publishes tile completions (no extra warps)
constexpr bool has_math_warps(int math) { return math >= 1 && math <= 3; }
constexpr int threads_of(int math) { return 32 * (kCtrlWarps + (has_math_warps(math) ? kFuseMathWarps : 0) + kEpiWarps); }

// One k-block is one 128-byte swizzle row of K (K-major) or one TMA box of k-rows (MN-major); fp16 pieces.
template <bool MN>
struct Geo {
    static constexpr int BK = 64;                        // K elements per k-block
    static constexpr int UK = 16;                        // K per tcgen05.mma
    static constexpr int BOX_MN = 64;                    // MN elements per 128-byte row of an MN-major box
    // K-major: rows of 128 B, 8-row groups 1024 B apart (SBO), LBO unused (= 1); a k-step is +32 B in the row.
    // MN-major: each k-row holds 128 B of MN; the next MN chunk is one TMA box (BK * 128 B) away (LBO); k-rows in
    //   groups of 8, 1024 B apart (SWIZZLE_128B); a k-step of UK rows is + UK * 128 B.
    static constexpr uint32_t kstep = MN ? UK * 128u : 32u;
    static constexpr uint32_t lbo = MN ? (BK * 128u) / 16u : 1u;
    static constexpr uint32_t sbo = 1024u / 16u;
    static constexpr uint32_t layout = 2u;               // SWIZZLE_128B
    // Instruction descriptor (cute::UMMA::InstrDescriptor): [4,6) D = F32 | [7,10) A fmt | [10,13) B fmt (0 = F16)
    // | 15 A major | 16 B major (1 = MN) | [17,23) N >> 3 | [24,29) M >> 4 (256 across the pair)
    static constexpr uint32_t idesc = (1u << 4) | (MN ? ((1u << 15) | (1u << 16)) : 0u) | ((uint32_t)(BN >> 3) << 17) |
                                      ((uint32_t)(256 >> 4) << 24);
    // measured shrink of a TMEM chunk sum per k-block of 12 truncating MMAs (see header)
    static constexpr float trunc_bias = 1.85e-7f;
    // k-blocks per TMEM chunk: every promotion costs 128 KiB of tcgen05.ld per CTA at ~64 B/clk, which stalls the
    // MMA stream; 4 keeps the rms error at 5e-7 (fp32 SGEMM: 1.1e-6 at K = 3993) for half the promotion traffic of 2
    static constexpr int default_kc = 4;
};

// EX names an operand that is EXACTLY representable as one fp16 piece (no lo plane): 1 = A, 2 = B.  The library's own
// Philox noise is drawn on the fp16 grid, so the forward (A = noise) and the backward (B = noise) products need only
// two MMA passes and three 16 KiB tiles per stage (48 KiB, 4-deep ring).
template <int EX>
struct Ring {
    static constexpr int NA = (EX == 1) ? 1 : 2, NB = (EX == 2) ? 1 : 2;       // planes staged per operand
    static constexpr int STAGE_BYTES = (NA + NB) * A_BYTES;                       // 64 KiB (EX = 0) or 48 KiB
    static constexpr int STAGES = (EX == 0) ? 3 : 4;
    static constexpr int RING_BYTES = STAGES * STAGE_BYTES;
    // measured truncation bias per k-block relative to the 3-pass constant: 1.30e-7 / 1.85e-7
    static constexpr float BIAS_SCALE = (EX == 0) ? 1.0f : 0.70f;
};
constexpr int kFusePaccBytes = kFuseMathWarps * 2 * 256 * (int)sizeof(float);   // 16 KiB: per math warp [2][256]
template <int EX>
constexpr int smem_bytes_of(int math) { return 1024 + Ring<EX>::RING_BYTES + BAR_BYTES + (math == 1 ? kFusePaccBytes : 0); }

// ------------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    const long long t0 = clock64();
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (!done && clock64() - t0 > 4000000000LL) __trap();   // ~2 s: a protocol bug must not hang the GPU
    } while (!done);
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 | [32,46) stride byte offset >> 4
//   [46,48) version = 1 (sm_100) | [61,64) layout type: 2 = SWIZZLE_128B (16 B atoms)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo16, uint32_t sbo16, uint32_t layout) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)(lbo16 & 0x3FFFu) << 16) | ((uint64_t)(sbo16 & 0x3FFFu) << 32) |
           (1ull << 46) | ((uint64_t)layout << 61);
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint32_t bar, uint16_t mask) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"(mask)
        : "memory");
}
__device__ __forceinline__ void tc_mma_2sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// Register re-partitioning between the warpgroups of a FUSE kernel (a warpgroup = 4 consecutive warps)
template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
// 896 threads x 72 registers at launch = 64512, re-dealt as 128 x 40 + 256 x 56 + 512 x 88 = 64512
constexpr int kRegCtrl = 40, kRegMath = 56, kRegEpi = 88;
static_assert(128 * kRegCtrl + 32 * kFuseMathWarps * kRegMath + 512 * kRegEpi <= 896 * 72, "register budget of the fused kernel");

// One thread's 64 consecutive output columns.  Rows whose start is not 16-byte aligned (odd ldc: g_R, the 512 -> L
// heads) get LEAD scalar stores up to the next 16-byte boundary, 15 vector stores, and the rest as scalars; every
// register index is a compile-time constant.
template <int LEAD>
__device__ __forceinline__ void store_row64(float* __restrict__ dst, const float (&acc)[64], float k) {
#pragma unroll
    for (int j = 0; j < LEAD; ++j) dst[j] = acc[j] * k;
    constexpr int NV = (LEAD == 0) ? 16 : 15;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
        const int j = LEAD + 4 * v;
        *reinterpret_cast<float4*>(dst + j) = make_float4(acc[j] * k, acc[j + 1] * k, acc[j + 2] * k, acc[j + 3] * k);
    }
#pragma unroll
    for (int j = LEAD + 4 * NV; j < 64; ++j) dst[j] = acc[j] * k;
}

// ------------------------------------------------------------------------------------------------ GEMM
// C[Mc, Nc] (row-major, pitch ldc) = inv_scale * sum_k A(m, k) * B(n, k); operands come pre-split as [2][.][.]
// planes (0 = hi, 1 = lo) through 3-D TMA maps.
//   MN == false: A is [Mc][K], B is [Nc][K] (K contiguous);   one box {BK, rows, 1} per tile and plane
//   MN == true : A is [K][Mc], B is [K][Nc] (Mc / Nc contiguous); boxes {BOX_MN, BK, 1}
// A cluster of two CTAs on neighbouring SMs owns a 256 x 256 tile.  Each CTA stages its own 128 rows of A and HALF of
// the B tile (128 of the 256 columns); the leader's single thread issues tcgen05.mma.cta_group::2 (M256 N256): the
// hardware reads A and B from both CTAs' shared memory and writes each CTA's 128 rows of D into its own tensor
// memory.  Barriers:
//   full[s]   (leader only)  armed by the leader with the bytes of BOTH CTAs; both CTAs' TMA loads complete_tx on it
//   empty[s]  (per CTA)      tcgen05.commit multicast to both CTAs
//   tfull[b]  (per CTA)      tcgen05.commit multicast to both CTAs
//   tempty[b] (leader only)  one arrive per promotion warp of both CTAs (remote arrive from the peer)
// Work items.  Tiles [0, full_tiles) fill whole waves of the persistent grid and run over all of K.  Each tile of the
// last, partial wave may be cut into `ksplit` slices of K so that the wave keeps every pair busy for 1/ksplit of a
// tile time instead of leaving most of them idle for a whole one: slice 0 writes C, slice j > 0 writes a 256 x 256
// scratch tile that tail_fixup_kernel adds to C afterwards (fixed order -> reproducible).
// store_cols: the epilogue writes columns [0, store_cols) of a row, Nc unless the caller owns the row padding up to ldc
// (the loss path's 16-byte rows, capi.cu) and lets the last 64-column block of a row go out as 16-byte stores.
struct GemmArgs {
    float* C;
    int Mc, Nc, K, ldc, store_cols, tiles_m, tiles_n, kc;
    const uint32_t *absmax_a, *absmax_b;
    int full_tiles, ksplit;
    float* partials;
};

// MATH: what the eight extra "math" warps of the CTA do (fused_rows.cuh): 0 = there are none, 1 = the probit row
// forward on finished tiles (opt-in), 2 = draw the Philox noise of the A operand just ahead of the tiles that read it,
// 3 = sum the finished tiles over the ranks of a data-parallel run through NVLink peer memory, 4 = no math warps, but
// finished tiles are published in peer memory for the exchange kernel that runs BESIDE this one on a few reserved SMs.
template <bool MN, int EX, int MATH, bool STABLE>
__global__ void __launch_bounds__(threads_of(MATH), 1)
gemm_split_2sm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs g,
                      const FuseFwd fz, const FuseNoise fnz, const FusePeer fpz) {
    constexpr bool FUSE = MATH >= 1 && MATH <= 3;
    constexpr bool PUBLISH = MATH == 3 || MATH == 4;
    using G = Geo<MN>;
    using R2 = Ring<EX>;
    constexpr int STAGES2 = R2::STAGES, STAGE2_BYTES = R2::STAGE_BYTES;
    constexpr int kFirstEpi = kCtrlWarps + (FUSE ? kFuseMathWarps : 0);
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;             // 128B-swizzled tiles need 1024 B alignment
    uint8_t* gen = smem_raw + (base - raw);
    const uint32_t bars = base + R2::RING_BYTES;
    // barrier slots (8 B each): full[STAGES], empty[STAGES], tfull[2], tempty[2]; then the TMEM base address
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (STAGES2 + s); };
    auto tfull_bar = [&](int a) { return bars + 8u * (2 * STAGES2 + a); };
    auto tempty_bar = [&](int a) { return bars + 8u * (2 * STAGES2 + 2 + a); };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen + R2::RING_BYTES + 128);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank() & 1u;             // position inside the pair (0 = leader)
    const bool leader = rank == 0;
    const int cluster = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
    const int num_tiles = g.tiles_m * g.tiles_n;
    const int num_items = (g.ksplit > 1) ? g.full_tiles + (num_tiles - g.full_tiles) * g.ksplit : num_tiles;
    struct Item { int st, kb_lo, kb_hi, slice; };
    auto item_of = [&](int w, int num_kb) {
        Item it;
        if (g.ksplit <= 1 || w < g.full_tiles) { it.st = w; it.kb_lo = 0; it.kb_hi = num_kb; it.slice = 0; return it; }
        const int r = w - g.full_tiles;
        it.st = g.full_tiles + r / g.ksplit;
        it.slice = r % g.ksplit;
        it.kb_lo = (int)(((long long)num_kb * it.slice) / g.ksplit);
        it.kb_hi = (int)(((long long)num_kb * (it.slice + 1)) / g.ksplit);
        return it;
    };
    if (threadIdx.x == 0) {
        if (PUBLISH) {   // the peer exchange's watermark and the promotion warps' arrival count
            *reinterpret_cast<volatile int*>(gen + R2::RING_BYTES + 192) = 0;
            *reinterpret_cast<volatile int*>(gen + R2::RING_BYTES + 196) = 0;
        }
        for (int s = 0; s < STAGES2; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 2 * kEpiWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)),
                     "r"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                       // peer barriers are initialised before anyone signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int num_kb = (g.K + G::BK - 1) / G::BK;

    if (warp < kCtrlWarps) {
        if (FUSE) reg_dec<kRegCtrl>();
        if (warp == 0 && lane == 0) {   // ------------------------------------------------ TMA producer (every CTA)
            int stage = 0, noise_block = -1;
            uint32_t phase = 0;
            for (int w = cluster; w < num_items; w += num_clusters) {
                const Item it = item_of(w, num_kb);
                const int m0 = (it.st / g.tiles_n) * 256 + (int)rank * BM;     // this CTA's 128 rows of A
                const int n0 = (it.st % g.tiles_n) * BN + (int)rank * HB;      // this CTA's half of the B tile
                if (MATH == 2 && (m0 >> 7) != noise_block && m0 < g.Mc) {      // the math warps of the grid draw these rows
                    noise_block = m0 >> 7;
                    noise_wait_block(fnz.ready + noise_block, (unsigned)(gridDim.x * kFuseMathWarps));
                }
                for (int kb = it.kb_lo; kb < it.kb_hi; ++kb) {
                    mbar_wait(empty_bar(stage), phase ^ 1u);
                    const uint32_t fb = map_to_cta(full_bar(stage), 0);        // the leader's barrier collects both CTAs' bytes
                    if (leader) mbar_arrive_expect_tx(full_bar(stage), 2 * STAGE2_BYTES);
                    const uint32_t sa = base + stage * STAGE2_BYTES, sb = sa + R2::NA * A_BYTES;
                    if (!MN) {
#pragma unroll
                        for (int pl = 0; pl < R2::NA; ++pl) tma_load_3d_2sm(sa + pl * A_BYTES, &tmA, fb, kb * G::BK, m0, pl);
#pragma unroll
                        for (int pl = 0; pl < R2::NB; ++pl) tma_load_3d_2sm(sb + pl * A_BYTES, &tmB, fb, kb * G::BK, n0, pl);
                    } else {
                        // MN-major tiles are BOX_MN-wide column boxes of BK k-rows
                        constexpr int box = G::BK * 128;
#pragma unroll
                        for (int j = 0; j < BM / G::BOX_MN; ++j)
#pragma unroll
                            for (int pl = 0; pl < R2::NA; ++pl)
                                tma_load_3d_2sm(sa + pl * A_BYTES + j * box, &tmA, fb, m0 + j * G::BOX_MN, kb * G::BK, pl);
#pragma unroll
                        for (int j = 0; j < HB / G::BOX_MN; ++j)
#pragma unroll
                            for (int pl = 0; pl < R2::NB; ++pl)
                                tma_load_3d_2sm(sb + pl * A_BYTES + j * box, &tmB, fb, n0 + j * G::BOX_MN, kb * G::BK, pl);
                    }
                    if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
                }
            }
        } else if (warp == 1 && lane == 0 && leader) {   // --------------------------------- MMA issuer (leader CTA only)
            int stage = 0, buf = 0;
            uint32_t phase = 0, bphase = 0;
            for (int w = cluster; w < num_items; w += num_clusters) {
                const Item it = item_of(w, num_kb);
                for (int kb0 = it.kb_lo; kb0 < it.kb_hi; kb0 += g.kc) {
                    mbar_wait(tempty_bar(buf), bphase ^ 1u);     // both CTAs' promotion warps have drained this buffer
                    tc_fence_after();
                    const uint32_t d = tmem_base + (uint32_t)(buf * BN);
                    const int kb1 = min(kb0 + g.kc, it.kb_hi);
                    for (int kb = kb0; kb < kb1; ++kb) {
                        mbar_wait(full_bar(stage), phase);
                        tc_fence_after();
                        const uint32_t sa = base + stage * STAGE2_BYTES, sb = sa + R2::NA * A_BYTES;
#pragma unroll
                        for (int kk = 0; kk < G::BK / G::UK; ++kk) {
                            const uint32_t first = (kb != kb0 || kk != 0) ? 1u : 0u;
                            const uint64_t a_hi = umma_desc(sa + kk * G::kstep, G::lbo, G::sbo, G::layout);
                            const uint64_t b_hi = umma_desc(sb + kk * G::kstep, G::lbo, G::sbo, G::layout);
                            if (EX == 1) {          // A exact: A.B_lo + A.B_hi
                                const uint64_t b_lo = umma_desc(sb + A_BYTES + kk * G::kstep, G::lbo, G::sbo, G::layout);
                                tc_mma_2sm(d, a_hi, b_lo, G::idesc, first);
                            } else if (EX == 2) {   // B exact: A_lo.B + A_hi.B
                                const uint64_t a_lo = umma_desc(sa + A_BYTES + kk * G::kstep, G::lbo, G::sbo, G::layout);
                                tc_mma_2sm(d, a_lo, b_hi, G::idesc, first);
                            } else {                // small terms first
                                const uint64_t a_lo = umma_desc(sa + A_BYTES + kk * G::kstep, G::lbo, G::sbo, G::layout);
                                const uint64_t b_lo = umma_desc(sb + A_BYTES + kk * G::kstep, G::lbo, G::sbo, G::layout);
                                tc_mma_2sm(d, a_lo, b_hi, G::idesc, first);
                                tc_mma_2sm(d, a_hi, b_lo, G::idesc, 1u);
                            }
                            tc_mma_2sm(d, a_hi, b_hi, G::idesc, 1u);
                        }
                        tc_commit_2sm(empty_bar(stage), 3);      // the stage is reusable in both CTAs once these MMAs retire
                        if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
                    }
                    tc_commit_2sm(tfull_bar(buf), 3);            // chunk complete in both CTAs' tensor memory
                    if (++buf == 2) { buf = 0; bphase ^= 1u; }
                }
            }
        } else if (PUBLISH && warp == 3 && lane == 0) {   // --------------------------------- tile publisher
            int n = 0;
            for (int w = cluster; w < num_items; w += num_clusters) {
                const Item it = item_of(w, num_kb);
                if (it.slice == 0 && it.st < fpz.full_tiles)
                    peer_publish_tile(fpz, reinterpret_cast<volatile int*>(gen + R2::RING_BYTES + 196), n++, it.st);
            }
        }
    } else if (FUSE && warp < kFirstEpi) {   // ------------------- math warps
        reg_dec<kRegMath>();
        const int mw = warp - kCtrlWarps;
        if (MATH == 1) {         // row math of the probit forward on finished tiles
            float* pacc = reinterpret_cast<float*>(gen + R2::RING_BYTES + BAR_BYTES) + mw * 512;
            fuse_math_loop<STABLE>(fz, cluster, num_clusters, num_tiles, g.tiles_n, (int)rank * kFuseMathWarps + mw, pacc, lane);
        } else if (MATH == 2) {  // the A operand's Philox noise, just ahead of the tiles
            noise_math_loop(fnz, (int)blockIdx.x * kFuseMathWarps + mw, (int)gridDim.x * kFuseMathWarps, lane);
        } else {                 // this rank's tiles of the sum over the ranks
            peer_math_loop(fpz, (int)blockIdx.x, (int)gridDim.x, mw, lane, reinterpret_cast<volatile int*>(gen + R2::RING_BYTES + 192));
        }
    } else {   // --------------------------------------------------- promotion + epilogue (both CTAs, own 128 rows)
        if (FUSE) reg_inc<kRegEpi>();
        const int q = warp & 3, h = (warp - kFirstEpi) >> 2;      // TMEM lane quadrant = warp id mod 4
        // 1 / (s_a * s_b) as two powers of two (common.cuh): exact for every normal result; extra == 1 unless the two
        // scales together leave the fp32 exponent range
        const Descale ds = descale_from_absmax_bits(g.absmax_a ? *g.absmax_a : 0u, g.absmax_b ? *g.absmax_b : 0u);
        const float inv_scale = ds.main;
        const bool vec_store = (g.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(g.C) & 15u) == 0;
        float acc[64];
#pragma unroll
        for (int j = 0; j < 64; ++j) acc[j] = 0.0f;
        int buf = 0;
        uint32_t bphase = 0;
        for (int w = cluster; w < num_items; w += num_clusters) {
            const Item it = item_of(w, num_kb);
            const int st = it.st;
            for (int kb0 = it.kb_lo; kb0 < it.kb_hi; kb0 += g.kc) {
                mbar_wait(tfull_bar(buf), bphase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + h * 64);
                const float unbias = 1.0f + G::trunc_bias * R2::BIAS_SCALE * (float)(min(kb0 + g.kc, it.kb_hi) - kb0);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    uint32_t v[16];
                    tmem_ld_32x16(taddr + i * 16, v);
#pragma unroll
                    for (int j = 0; j < 16; ++j)   // round-to-nearest promotion
                        acc[i * 16 + j] = fmaf(__uint_as_float(v[j]), unbias, acc[i * 16 + j]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(map_to_cta(tempty_bar(buf), 0));
                if (++buf == 2) { buf = 0; bphase ^= 1u; }
            }
            const int row = (st / g.tiles_n) * 256 + (int)rank * BM + q * 32 + lane;
            const int col0 = (st % g.tiles_n) * BN + h * 64;
            if (ds.extra != 1.0f) {   // extreme operand scales only (uniform over the CTA)
#pragma unroll
                for (int j = 0; j < 64; ++j) acc[j] *= ds.extra;
            }
            if (it.slice > 0) {
                // K-slice of a tail tile: the whole 256 x 256 scratch tile is written (rows / columns beyond the
                // matrix hold sums of zero-filled boxes, i.e. zeros)
                float* __restrict__ prow = g.partials + ((size_t)(st - g.full_tiles) * (g.ksplit - 1) + (it.slice - 1)) * (256 * BN) +
                                           (size_t)((int)rank * BM + q * 32 + lane) * BN + h * 64;
#pragma unroll
                for (int j = 0; j < 64; j += 4)
                    *reinterpret_cast<float4*>(prow + j) =
                        make_float4(acc[j] * inv_scale, acc[j + 1] * inv_scale, acc[j + 2] * inv_scale, acc[j + 3] * inv_scale);
            } else if (row < g.Mc && col0 < g.Nc) {
                float* __restrict__ crow = g.C + (size_t)row * g.ldc;
                if (vec_store && col0 + 64 <= g.store_cols) {
                    // 16-byte stores: rows are 16 B aligned (ldc % 4 == 0); columns in [Nc, store_cols) are padding
                    // the caller owns
#pragma unroll
                    for (int j = 0; j < 64; j += 4)
                        *reinterpret_cast<float4*>(crow + col0 + j) =
                            make_float4(acc[j] * inv_scale, acc[j + 1] * inv_scale, acc[j + 2] * inv_scale, acc[j + 3] * inv_scale);
                } else if (col0 + 64 <= g.Nc) {
                    // unaligned row: scalars up to the next 16-byte boundary, then vectors
                    float* __restrict__ d = crow + col0;
                    switch ((4 - (int)((reinterpret_cast<uintptr_t>(d) >> 2) & 3u)) & 3) {
                        case 0: store_row64<0>(d, acc, inv_scale); break;
                        case 1: store_row64<1>(d, acc, inv_scale); break;
                        case 2: store_row64<2>(d, acc, inv_scale); break;
                        default: store_row64<3>(d, acc, inv_scale); break;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 64; ++j)
                        if (col0 + j < g.Nc) crow[col0 + j] = acc[j] * inv_scale;
                }
            }
            if (MATH == 1) fuse_signal_tile(fz.done, st, lane);   // this warp's part of the tile is in memory
            if (PUBLISH && it.slice == 0 && st < fpz.full_tiles)
                peer_arrive_tile(reinterpret_cast<volatile int*>(gen + R2::RING_BYTES + 196), lane);
#pragma unroll
            for (int j = 0; j < 64; ++j) acc[j] = 0.0f;
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                       // the peer may still be reading our smem / signalling us
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// C += the K-slices 1 .. ksplit-1 of the tail tiles (see above), slice order fixed.  64 CTAs per tail tile, each 4 rows
// of 256 columns; the loads of a thread's four rows are independent of each other.
__global__ void __launch_bounds__(256)
tail_fixup_kernel(float* __restrict__ C, int Mc, int Nc, int ldc, int tiles_n, int full_tiles, int ksplit,
                  const float* __restrict__ partials) {
    const int t = blockIdx.x >> 6, rows0 = (blockIdx.x & 63) * 4;
    const int st = full_tiles + t;
    const int m0 = (st / tiles_n) * 256, n0 = (st % tiles_n) * BN;
    const float* __restrict__ p = partials + (size_t)t * (ksplit - 1) * (256 * BN);
    const int c = threadIdx.x;                      // BN == 256 columns, one per thread
    if (n0 + c >= Nc) return;
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = (m0 + rows0 + i < Mc) ? C[(size_t)(m0 + rows0 + i) * ldc + n0 + c] : 0.0f;
    for (int j = 0; j < ksplit - 1; ++j) {
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] += p[(size_t)j * (256 * BN) + (rows0 + i) * BN + c];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (m0 + rows0 + i < Mc) C[(size_t)(m0 + rows0 + i) * ldc + n0 + c] = v[i];
}

// ------------------------------------------------------------------------------------------------ pre-passes
// |x| as raw fp32 bits, 0 for Inf and NaN
__device__ __forceinline__ uint32_t finite_abs_bits(uint32_t b) {
    b &= 0x7FFFFFFFu;
    return b < 0x7F800000u ? b : 0u;
}

// max |x| over the FINITE elements as raw fp32 bits (ordering of non-negative floats == ordering of their bit
// patterns): an Inf or NaN element must not cost the finite ones their scale
__global__ void __launch_bounds__(256)
absmax_kernel(const float* __restrict__ src, size_t n, uint32_t* __restrict__ out) {
    uint32_t m = 0;
    const size_t tid = blockIdx.x * (size_t)blockDim.x + threadIdx.x, nthr = (size_t)gridDim.x * blockDim.x;
    size_t done = 0;
    if ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) {      // 16-byte loads over the aligned bulk
        const size_t n4 = n / 4;
        const uint4* __restrict__ s4 = reinterpret_cast<const uint4*>(src);
        for (size_t i = tid; i < n4; i += nthr) {
            const uint4 v = s4[i];
            const uint32_t a = max(max(finite_abs_bits(v.x), finite_abs_bits(v.y)), max(finite_abs_bits(v.z), finite_abs_bits(v.w)));
            m = a > m ? a : m;
        }
        done = n4 * 4;
    }
    for (size_t i = done + tid; i < n; i += nthr) {
        const uint32_t b = finite_abs_bits(__float_as_uint(src[i]));
        m = b > m ? b : m;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const uint32_t t = __shfl_xor_sync(0xffffffffu, m, o);
        m = t > m ? t : m;
    }
    // one atomic per CTA: thousands of atomics on one address serialise (10 us for a 5 MB tensor with one per warp)
    __shared__ uint32_t s_m[8];
    if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) m = s_m[w] > m ? s_m[w] : m;
        if (m != 0) atomicMax(out, m);
    }
}

// hi = fp16(x * s), lo = fp16(x * s - hi) with s from the tensor's absmax; lo = 0 where x is infinite (Inf - Inf
// would make it NaN; x * s of a finite x stays below 2^15); four elements per thread.  dst planes are
// [rows][dpitch], pad columns zero.  perm_S > 0: the source rows are s-major (r = s * perm_B + b, the (S, B, Z) noise
// tensor of mpvae.py:162) and are written b-major (b * perm_S + s), the row order of the loss path's products.
__global__ void __launch_bounds__(256)
split_f16_kernel(const float* __restrict__ src, __half* __restrict__ dst, int rows, int cols, int spitch, int dpitch,
                 size_t plane, const uint32_t* __restrict__ absmax, int perm_S, int perm_B) {
    const float s = absmax ? scale_from_absmax_bits(*absmax) : 1.0f;
    const size_t n4 = (size_t)rows * dpitch / 4;          // dpitch is a multiple of 64: groups of 4 never straddle rows
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        const size_t e = 4 * i;
        const int r = (int)(e / dpitch), c = (int)(e % dpitch);
        const float* __restrict__ sp = src + (size_t)r * spitch + c;
        float x[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) x[j] = (c + j < cols) ? sp[j] * s : 0.0f;
        __half h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            h[j] = __float2half_rn(x[j]);
            l[j] = __hisinf(h[j]) ? __float2half_rn(0.0f) : __float2half_rn(x[j] - __half2float(h[j]));
        }
        const __half2 h01 = __halves2half2(h[0], h[1]), h23 = __halves2half2(h[2], h[3]);
        const __half2 l01 = __halves2half2(l[0], l[1]), l23 = __halves2half2(l[2], l[3]);
        uint2 hv, lv;
        hv.x = *reinterpret_cast<const uint32_t*>(&h01); hv.y = *reinterpret_cast<const uint32_t*>(&h23);
        lv.x = *reinterpret_cast<const uint32_t*>(&l01); lv.y = *reinterpret_cast<const uint32_t*>(&l23);
        const int rd = perm_S > 0 ? (r % perm_B) * perm_S + r / perm_B : r;
        const size_t o = (size_t)rd * dpitch + c;
        *reinterpret_cast<uint2*>(dst + o) = hv;
        *reinterpret_cast<uint2*>(dst + plane + o) = lv;
    }
}

// ------------------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 3-D map over a split operand [planes][rows][pitch] of halves: dims {cols, rows, planes}, 128B swizzle, zero OOB fill.
int make_map(CUtensorMap* map, const void* ptr, int cols, int rows, int pitch, int box_cols, int box_rows, int planes = 2) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled unavailable from the driver"); return 8; }
    const cuuint64_t esz = 2;
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)planes};
    cuuint64_t strides[2] = {(cuuint64_t)pitch * esz, (cuuint64_t)rows * pitch * esz};
    cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d) cols=%d rows=%d pitch=%d", (int)r, cols, rows, pitch); return 8; }
    return 0;
}

int pitch_of(int cols) { return ceil_div(cols, 64) * 64; }

// MPVAE_TC_KC: TMEM chunk length in k-blocks (accuracy / speed experiments, profiles/r01_exact_operand_kc_sweep.jsonl)
int chunk_kblocks(int dflt) {
    static int kc = -1;
    if (kc < 0) {
        const char* e = getenv("MPVAE_TC_KC");
        kc = e ? atoi(e) : 0;
    }
    return kc > 0 ? kc : dflt;
}

int grid_for(size_t n) { return (int)((n + 255) / 256 < (size_t)(8 * kNumSMs) ? (n + 255) / 256 : 8 * kNumSMs); }

// scratch layout of the all-in-one entry points: [absmax_a, absmax_b (256 B)] [A planes] [B planes] [tail scratch]
struct Scratch { uint32_t* absmax; char* a; char* b; };

size_t planes_bytes(size_t rows, size_t pitch) { return align_up(2 * rows * pitch * 2, 1024); }

Scratch carve_scratch(void* ws, size_t rows_a, size_t pitch_a) {
    char* p = static_cast<char*>(ws);
    return {reinterpret_cast<uint32_t*>(p), p + 256, p + 256 + planes_bytes(rows_a, pitch_a)};
}

// per-device one-time configuration (the attribute and the occupancy are per device / context)
constexpr int kMaxDevices = 64;
int current_device() {
    int d = 0;
    cudaGetDevice(&d);
    return (d >= 0 && d < kMaxDevices) ? d : 0;
}

template <bool MN, int EX, int MATH, bool STABLE>
int launch_gemm_2sm(const CUtensorMap& a, const CUtensorMap& b, GemmArgs g, const FuseFwd& fz, const FuseNoise& fnz,
                    cudaStream_t stream, size_t partials_bytes, FusePeer fpz = FusePeer{}, int* exchanged_tiles = nullptr) {
    auto kernel = gemm_split_2sm_kernel<MN, EX, MATH, STABLE>;
    static int max_clusters[kMaxDevices] = {};     // co-resident clusters (a cluster must fit inside one GPC)
    constexpr int smem = smem_bytes_of<EX>(MATH);
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.blockDim = dim3(threads_of(MATH));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const int dev = current_device();
    if (max_clusters[dev] == 0) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(gemm_split_2sm): %s", cudaGetErrorString(e)); return 4; }
        cfg.gridDim = dim3(kNumSMs / 2 * 2);
        int n = 0;
        e = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
        if (e != cudaSuccess || n <= 0) { set_error("cudaOccupancyMaxActiveClusters: %s", cudaGetErrorString(e)); return 4; }
        max_clusters[dev] = n < kNumSMs / 2 ? n : kNumSMs / 2;
    }
    // MATH == 4: a few SM pairs are left to the exchange kernel that runs beside this one (peer_reduce.cu)
    const int mc = max_clusters[dev] - (MATH == 4 ? exchange_sms(fpz.world) / 2 : 0);
    const int tiles = g.tiles_m * g.tiles_n;
    // K-split of the last, partial wave: worth it when the wave would leave at least half of the pairs idle and the
    // caller gave scratch for the slices
    g.full_tiles = tiles;
    g.ksplit = 1;
    static const bool no_split = getenv("MPVAE_TC_NO_KSPLIT") != nullptr;
    if (MATH != 1 && g.partials != nullptr && !no_split) {
        const int tail = tiles % mc, num_kb = ceil_div(g.K, Geo<MN>::BK);
        if (tail > 0) {
            // f slices per tail tile: the tail then takes ceil(tail * f / mc) / f of a tile time instead of a whole one;
            // the smallest f with the smallest cost, as long as a slice keeps a full TMEM chunk and the scratch holds it
            int best = 1;
            double best_cost = 1.0;
            for (int f = 2; f <= 8; ++f) {
                if (f > num_kb / g.kc) break;
                if ((size_t)tail * (f - 1) * 256 * BN * sizeof(float) > partials_bytes) break;
                const double cost = (double)ceil_div(tail * f, mc) / f;
                if (cost < best_cost - 1e-9) { best_cost = cost; best = f; }
            }
            if (best >= 2) { g.full_tiles = tiles - tail; g.ksplit = best; }
        }
    }
    const int items = g.full_tiles + (tiles - g.full_tiles) * g.ksplit;
    const int clusters = items < mc ? items : mc;
    cfg.gridDim = dim3(2 * clusters);
    if (MATH == 3 || MATH == 4) {
        // the K-sliced tail tiles are complete only after tail_fixup_kernel: they are exchanged after this kernel
        fpz.full_tiles = g.full_tiles;
        fpz.tiles_n = g.tiles_n;
        if (exchanged_tiles) *exchanged_tiles = g.full_tiles;
    }
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, a, b, g, fz, fnz, fpz);
    if (e != cudaSuccess) { set_error("gemm_split_2sm_kernel launch: %s", cudaGetErrorString(e)); return 3; }
    if (int rc = check_launch("gemm_split_2sm_kernel")) return rc;
    if (g.ksplit > 1) {
        static_assert(BN == 256, "tail_fixup_kernel maps one thread to one tile column");
        tail_fixup_kernel<<<(tiles - g.full_tiles) * 64, 256, 0, stream>>>(g.C, g.Mc, g.Nc, g.ldc, g.tiles_n, g.full_tiles, g.ksplit,
                                                                          g.partials);
        return check_launch("tail_fixup_kernel");
    }
    return 0;
}

// ex: 0 = both operands carry hi|lo planes, 1 = A is exact (single plane), 2 = B is exact
template <bool MN>
int launch_gemm(const CUtensorMap& a, const CUtensorMap& b, float* C, int Mc, int Nc, int K, int ldc, const uint32_t* ma,
                const uint32_t* mb, cudaStream_t stream, int ex, float* partials, size_t partials_bytes,
                const FuseFwd* fuse = nullptr, const FuseNoise* noise = nullptr, const FusePeer* peer = nullptr,
                int* exchanged_tiles = nullptr, int peer_mode = 3, bool write_pad = false) {
    GemmArgs g{};
    g.C = C; g.Mc = Mc; g.Nc = Nc; g.K = K; g.ldc = ldc;
    g.store_cols = write_pad ? ldc : Nc;
    g.tiles_m = ceil_div(Mc, 256); g.tiles_n = ceil_div(Nc, BN);
    // k-blocks per TMEM chunk: the same number of truncating MMAs per chunk (48) whether a k-step is 3 or 2 MMAs
    g.kc = chunk_kblocks(ex == 0 ? Geo<MN>::default_kc : (Geo<MN>::default_kc * 3) / 2);
    g.absmax_a = ma; g.absmax_b = mb;
    g.partials = partials;
    const FuseFwd none{};
    const FuseNoise nonoise{};
    if (peer != nullptr) {
        if (!MN || ex == 1 || fuse != nullptr || noise != nullptr) { set_error("fused exchange: tn products only"); return 7; }
        if (peer_mode == 4) {
            if (ex == 2) return launch_gemm_2sm<true, 2, 4, false>(a, b, g, none, nonoise, stream, partials_bytes, *peer, exchanged_tiles);
            return launch_gemm_2sm<true, 0, 4, false>(a, b, g, none, nonoise, stream, partials_bytes, *peer, exchanged_tiles);
        }
        if (ex == 2) return launch_gemm_2sm<true, 2, 3, false>(a, b, g, none, nonoise, stream, partials_bytes, *peer, exchanged_tiles);
        return launch_gemm_2sm<true, 0, 3, false>(a, b, g, none, nonoise, stream, partials_bytes, *peer, exchanged_tiles);
    }
    if (noise != nullptr) {
        if (MN || ex != 1 || fuse != nullptr) { set_error("just-in-time noise: nt products with an exact A operand only"); return 7; }
        return launch_gemm_2sm<false, 1, 2, false>(a, b, g, none, *noise, stream, 0);
    }
    if (fuse != nullptr) {
        if (MN || ex == 2) { set_error("fused forward: nt products only"); return 7; }
        if (fuse->stable) {
            if (ex == 1) return launch_gemm_2sm<false, 1, 1, true>(a, b, g, *fuse, nonoise, stream, 0);
            return launch_gemm_2sm<false, 0, 1, true>(a, b, g, *fuse, nonoise, stream, 0);
        }
        if (ex == 1) return launch_gemm_2sm<false, 1, 1, false>(a, b, g, *fuse, nonoise, stream, 0);
        return launch_gemm_2sm<false, 0, 1, false>(a, b, g, *fuse, nonoise, stream, 0);
    }
    if (ex == 1) return launch_gemm_2sm<MN, 1, 0, false>(a, b, g, none, nonoise, stream, partials_bytes);
    if (ex == 2) return launch_gemm_2sm<MN, 2, 0, false>(a, b, g, none, nonoise, stream, partials_bytes);
    return launch_gemm_2sm<MN, 0, 0, false>(a, b, g, none, nonoise, stream, partials_bytes);
}

}  // namespace

bool tc_available() { return true; }

int exchange_sms(int world) {
    // measured on 8 B200s (eurlex weak scaling, loss step; profiles/r02_fused_exchange.md): 8 SMs 1.85 ms, 16 SMs 1.73 - 1.83 ms,
    // 20 SMs 1.73 ms, 24 SMs 1.76 ms, 32 SMs 1.80 ms (exchange behind the product: 1.95 ms).  20 SMs leave 64 CTA pairs:
    // the 256 tiles of the eurlex g_R are then exactly four waves, no K-sliced tail.  On 2 GPUs, where each rank moves
    // less, 8 SMs are enough.
    static int forced = -1;
    if (forced < 0) {
        const char* e = getenv("MPVAE_EXCHANGE_SMS");
        forced = e ? atoi(e) : 0;
        if (forced != 0) forced = (forced < 2 ? 2 : forced > 64 ? 64 : forced) & ~1;
    }
    return forced != 0 ? forced : (world > 2 ? 20 : 8);
}

// [absmax slots] [A planes] [B planes] [tail-wave scratch]
size_t tc_workspace_nt(int M, int N, int K) {
    const size_t kp = pitch_of(K);
    return 256 + planes_bytes(M, kp) + planes_bytes(N, kp) + tc_tail_scratch_bytes();
}

size_t tc_workspace_tn(int M, int N1, int N2) {
    return 256 + planes_bytes(M, pitch_of(N1)) + planes_bytes(M, pitch_of(N2)) + tc_tail_scratch_bytes();
}

int tc_split(const float* src, int rows, int cols, void* planes, uint32_t* absmax, int compute_absmax, cudaStream_t stream,
             int src_pitch, int perm_S, int perm_B) {
    if (src_pitch <= 0) src_pitch = cols;
    const int pitch = pitch_of(cols);
    const size_t n = (size_t)rows * pitch;
    if (perm_S > 0 && (long long)perm_S * perm_B != rows) { set_error("tc_split: row permutation %d x %d != %d rows", perm_S, perm_B, rows); return 1; }
    if (absmax && compute_absmax) {
        absmax_kernel<<<grid_for((size_t)rows * cols), 256, 0, stream>>>(src, (size_t)rows * cols, absmax);
        if (int rc = check_launch("absmax_kernel")) return rc;
    }
    split_f16_kernel<<<grid_for(n / 4), 256, 0, stream>>>(src, static_cast<__half*>(planes), rows, cols, src_pitch, pitch, n, absmax,
                                                         perm_S, perm_B);
    return check_launch("split_f16_kernel");
}

int tc_contract_nt(const float* A, const float* Bm, float* C, int M, int N, int K, void* ws, size_t ws_bytes,
                   cudaStream_t stream, int reuse_planes, int exact, int ldc, int allow_ksplit) {
    if (!ws || ws_bytes < tc_workspace_nt(M, N, K)) { set_error("tc_contract_nt: workspace too small"); return 5; }
    if (ldc <= 0) ldc = N;
    const int ex = exact ? 1 : 0;
    const int kp = pitch_of(K);
    const Scratch s = carve_scratch(ws, M, kp);
    if (!reuse_planes) {
        if (cudaMemsetAsync(s.absmax, 0, 256, stream) != cudaSuccess) { set_error("cudaMemsetAsync failed"); return 2; }
        if (int rc = tc_split(A, M, K, s.a, s.absmax, 1, stream)) return rc;
        if (int rc = tc_split(Bm, N, K, s.b, s.absmax + 1, 1, stream)) return rc;
    }
    // K-sliced partial waves only on request: without them each element's summation order is a function of K alone,
    // which the loss path needs (a row's predictions must not depend on how many rows the call holds)
    void* tail = allow_ksplit ? static_cast<void*>(s.b + planes_bytes(N, kp)) : nullptr;
    return tc_gemm_nt(s.a, s.b, C, M, N, K, s.absmax, s.absmax + 1, stream, ldc, ex, tail, allow_ksplit ? tc_tail_scratch_bytes() : 0);
}

int tc_contract_tn(const float* A, const float* Bm, float* C, int M, int N1, int N2, void* ws, size_t ws_bytes,
                   cudaStream_t stream, int reuse_planes, int exact) {
    if (!ws || ws_bytes < tc_workspace_tn(M, N1, N2)) { set_error("tc_contract_tn: workspace too small"); return 5; }
    const int p1 = pitch_of(N1), p2 = pitch_of(N2);
    const Scratch s = carve_scratch(ws, M, p1);
    if (!reuse_planes) {
        if (cudaMemsetAsync(s.absmax, 0, 256, stream) != cudaSuccess) { set_error("cudaMemsetAsync failed"); return 2; }
        if (int rc = tc_split(A, M, N1, s.a, s.absmax, 1, stream)) return rc;
        if (int rc = tc_split(Bm, M, N2, s.b, s.absmax + 1, 1, stream)) return rc;
    }
    return tc_gemm_tn(s.a, s.b, C, M, N1, N2, s.absmax, s.absmax + 1, stream, exact ? 1 : 0, s.b + planes_bytes(M, p2),
                      tc_tail_scratch_bytes());
}

// ------------------------------------------------------------------------------------------------ staged interface
size_t tc_planes_bytes(int rows, int cols) { return planes_bytes((size_t)rows, (size_t)pitch_of(cols)); }

namespace {

// Philox normals written straight into ONE operand plane (scale 1: |n| < 6 fits fp16; the values lie on the fp16 grid,
// so there is no lo piece).  One thread per counter, same counter -> element mapping as philox_normal_kernel, so the
// numbers are identical to the fp32 tensor it would write.  Plane rows are b-major: element (s, b, z) -> row b*S + s.
__global__ void __launch_bounds__(256)
philox_planes_kernel(__half* __restrict__ planes, int S, int B, int Z, int pitch, int Bg, int row0, uint2 key, uint2 off,
                     const unsigned long long* __restrict__ off_dev) {
    const int s = blockIdx.y;
    const unsigned long long span_beg = ((unsigned long long)s * Bg + row0) * Z;
    const unsigned long long span_end = span_beg + (unsigned long long)B * Z;
    const unsigned long long c = (span_beg >> 2) + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if ((c << 2) >= span_end) return;
    float n[4];
    philox_normal4(c, key, philox_offset(off, off_dev), n);
    // position of flat index 4c inside this sample's (B, Z) block (B * Z < 2^31 is checked by the launcher);
    // one 32-bit division per thread, then walk the four elements
    const long long e0 = (long long)((c << 2) - span_beg);               // may be -3..-1 for the first counter
    int row = e0 >= 0 ? (int)((unsigned)e0 / (unsigned)Z) : -1;
    int col = e0 >= 0 ? (int)((unsigned)e0 % (unsigned)Z) : Z + (int)e0;
    if (row >= 0 && row < B && col + 4 <= Z) {
        // the common case: four neighbours of one row; as few stores as the alignment of the destination allows
        // (it is the same for every thread of a row, so a warp does not diverge here)
        __half* dst = planes + ((size_t)row * S + s) * pitch + (size_t)col;
        const __half2 p01 = __floats2half2_rn(n[0], n[1]), p23 = __floats2half2_rn(n[2], n[3]);
        const uintptr_t a = reinterpret_cast<uintptr_t>(dst);
        if ((a & 7u) == 0) {
            uint2 v;
            v.x = *reinterpret_cast<const uint32_t*>(&p01);
            v.y = *reinterpret_cast<const uint32_t*>(&p23);
            *reinterpret_cast<uint2*>(dst) = v;
        } else if ((a & 3u) == 0) {
            *reinterpret_cast<__half2*>(dst) = p01;
            *reinterpret_cast<__half2*>(dst + 2) = p23;
        } else {
            dst[0] = __low2half(p01);
            *reinterpret_cast<__half2*>(dst + 1) = __halves2half2(__high2half(p01), __low2half(p23));
            dst[3] = __high2half(p23);
        }
        return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int r = row, cc = col;
        if (++col == Z) { col = 0; ++row; }
        if (r < 0 || r >= B) continue;
        planes[((size_t)r * S + s) * pitch + (size_t)cc] = __float2half_rn(n[j]);
    }
}

}  // namespace

int tc_philox_planes(void* planes, int S, int B, int Z, int Bg, int row0, uint64_t seed, uint64_t offset,
                     const uint64_t* offset_dev, cudaStream_t stream) {
    if (S > 65535) { set_error("philox: S=%d exceeds grid.y limit", S); return 6; }
    if ((long long)B * Z >= 0x7fffffffLL || Z < 4) { set_error("philox planes: B*Z=%lld, Z=%d out of range", (long long)B * Z, Z); return 6; }
    const unsigned long long counters = ((unsigned long long)B * Z + 3) / 4 + 1;
    dim3 grid((unsigned)((counters + 255) / 256), S);
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const uint2 off = make_uint2((uint32_t)offset, (uint32_t)(offset >> 32));
    philox_planes_kernel<<<grid, 256, 0, stream>>>(static_cast<__half*>(planes), S, B, Z, pitch_of(Z), Bg, row0, key, off,
                                                  reinterpret_cast<const unsigned long long*>(offset_dev));
    return check_launch("philox_planes_kernel");
}

int tc_pitch(int cols) { return pitch_of(cols); }
int tc_absmax(const float* src, size_t n, uint32_t* out_bits, cudaStream_t stream) {
    absmax_kernel<<<grid_for(n), 256, 0, stream>>>(src, n, out_bits);
    return check_launch("absmax_kernel");
}

// room for two extra K-slices of every tile of a partial wave (three slices per tile), or seven of a short one
size_t tc_tail_scratch_bytes() { return (size_t)(kNumSMs / 2 - 1) * 2 * 256 * BN * sizeof(float); }

int tc_gemm_nt(const void* a_planes, const void* b_planes, float* C, int M, int N, int K, const uint32_t* absmax_a,
               const uint32_t* absmax_b, cudaStream_t stream, int ldc, int a_exact, void* tail_scratch, size_t tail_scratch_bytes,
               const FuseFwd* fuse, const FuseNoise* noise, int write_pad) {
    if (ldc <= 0) ldc = N;
    const int kp = pitch_of(K);
    CUtensorMap ma, mb;
    if (int rc = make_map(&ma, a_planes, K, M, kp, 64, BM, a_exact ? 1 : 2)) return rc;
    if (int rc = make_map(&mb, b_planes, K, N, kp, 64, HB)) return rc;
    return launch_gemm<false>(ma, mb, C, M, N, K, ldc, absmax_a, absmax_b, stream, a_exact ? 1 : 0, static_cast<float*>(tail_scratch),
                              tail_scratch_bytes, fuse, noise, nullptr, nullptr, 3, write_pad != 0);
}

int tc_gemm_tn(const void* a_planes, const void* b_planes, float* C, int M, int N1, int N2, const uint32_t* absmax_a,
               const uint32_t* absmax_b, cudaStream_t stream, int b_exact, void* tail_scratch, size_t tail_scratch_bytes,
               int a_pitch, const FusePeer* peer, int* exchanged_tiles, int peer_mode) {
    // a_pitch > 0: A is a column range of wider planes (row slab of C): a_planes points at its first column
    const int p1 = a_pitch > 0 ? a_pitch : pitch_of(N1), p2 = pitch_of(N2);
    CUtensorMap ma, mb;
    if (int rc = make_map(&ma, a_planes, N1, M, p1, 64, 64)) return rc;
    if (int rc = make_map(&mb, b_planes, N2, M, p2, 64, 64, b_exact ? 1 : 2)) return rc;
    return launch_gemm<true>(ma, mb, C, N1, N2, M, N2, absmax_a, absmax_b, stream, b_exact ? 2 : 0, static_cast<float*>(tail_scratch),
                             tail_scratch_bytes, nullptr, nullptr, peer, exchanged_tiles, peer_mode);
}

}  // namespace mpv
