// Building blocks of the small-regime kernels (L, Z <= 128, L * Z <= 8192: one CTA per batch row), shared by the loss
// forward (probit_rows.cu::probit_small_fwd_kernel) and the prediction-only kernel (predict.cu), so that both stage R,
// draw the noise and contract it in exactly the same way.  predict.cu's row passes also take row_of from here.
#pragma once
#include "philox.cuh"
#include "rows.h"

namespace mpv {

// row index of (s, b) in the scratch matrices (RowArgs::row_sb / row_ss)
__device__ __forceinline__ size_t row_of(const RowArgs& a, int s, int b) { return (size_t)b * a.row_sb + (size_t)s * a.row_ss; }

struct SmallArgs {
    RowArgs a;
    const float* r;            // (L, Z) fp32
    int Z;
    const float* noise_ext;    // (S, B, Z) caller's noise or nullptr
    float* noise_out;          // (S, B, Z) fp32 copy kept for the backward, or nullptr (inference)
    float* nr_out;             // (S*B, ldn) kept for the backward, or nullptr
    int Bg, row0;
    uint2 key, off;
    const unsigned long long* off_dev;
    float* partial;            // backward: (B, L*Z) per-row contributions to g_R
};

static inline SmallArgs small_args(const RowArgs& a, const SmallNoise& n) {
    SmallArgs p{};
    p.a = a;
    p.r = n.r; p.Z = n.Z;
    p.noise_ext = n.noise_ext; p.noise_out = n.noise_out; p.nr_out = n.nr_out;
    p.Bg = n.Bg; p.row0 = n.row0;
    p.key = make_uint2((uint32_t)n.seed, (uint32_t)(n.seed >> 32));
    p.off = make_uint2((uint32_t)n.offset, (uint32_t)(n.offset >> 32));
    p.off_dev = reinterpret_cast<const unsigned long long*>(n.offset_dev);
    p.partial = n.partial;
    return p;
}

constexpr int kSmallThreads = 512;   // sixteen warps: a sample pair each per round
constexpr int kSmallWarps = kSmallThreads / 32;

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// R (L x Z fp32) -> shared memory Rs: one TMA bulk copy (cp.async.bulk + mbarrier) for the 16-byte multiple, plain
// loads for the last few floats.  Called by every thread of the CTA; returns whether the bulk copy was issued, which
// small_r_wait then waits for (the caller may load other things in between).
template <int NT>
__device__ __forceinline__ bool small_r_stage(float* Rs, const float* __restrict__ r, int L, int Z, unsigned long long* s_bar) {
    const int tid = threadIdx.x;
    const uint32_t bytes16 = ((uint32_t)(L * Z) * 4u) & ~15u;
    const bool bulk = bytes16 != 0 && (reinterpret_cast<uintptr_t>(r) & 15u) == 0;
    const uint32_t bar = smem_addr(s_bar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0 && bulk) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes16) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_addr(Rs)), "l"(r), "r"(bytes16), "r"(bar)
                     : "memory");
    }
    for (int i = (bulk ? (int)(bytes16 >> 2) : 0) + tid; i < L * Z; i += NT) Rs[i] = r[i];
    return bulk;
}

// waits for the bulk copy of small_r_stage; the caller's __syncthreads() then publishes the plain-loaded tail too
__device__ __forceinline__ void small_r_wait(bool bulk, unsigned long long* s_bar) {
    if (!bulk) return;
    const uint32_t bar = smem_addr(s_bar);
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred q;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 q, [%1], 0;\n\t"
            "selp.u32 %0, 1, 0, q;\n\t}"
            : "=r"(done)
            : "r"(bar)
            : "memory");
    }
}

// One warp: the noise of samples s0 and s0 + 1 (those below S) of batch row b into nzw[0 .. 2Z), either copied from the
// caller's tensor or drawn in registers (Philox4x32-10 + Box-Muller, the numbers of philox_normal).  The caller
// __syncwarp()s before reading nzw.
__device__ __forceinline__ void small_noise_pair(float* nzw, const SmallArgs& p, int s0, int b, uint2 off, int lane) {
    const int S = p.a.S, B = p.a.B, Z = p.Z;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int s = s0 + i;
        if (s >= S) break;
        if (p.noise_ext) {
            const float* src = p.noise_ext + ((size_t)s * B + b) * Z;
            for (int z = lane; z < Z; z += 32) nzw[i * Z + z] = src[z];
        } else {
            // the normals of (s, global row, 0 .. Z): counters flat0 / 4 .. (flat0 + Z - 1) / 4 of the global tensor
            const unsigned long long flat0 = ((unsigned long long)s * p.Bg + p.row0 + b) * Z;
            const unsigned long long c0 = flat0 >> 2, c1 = (flat0 + Z - 1) >> 2;
            for (unsigned long long c = c0 + lane; c <= c1; c += 32) {
                float n[4];
                philox_normal4(c, p.key, off, n);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const long long z = (long long)(c << 2) + j - (long long)flat0;
                    if (z >= 0 && z < Z) nzw[i * Z + z] = n[j];
                }
            }
        }
    }
}

// nr of label row rl (Z floats of R in shared memory) for the two samples in nzw: a warp-level FMA chain in k order (the
// chain of contract_fma.cu: bit-equal results)
__device__ __forceinline__ void small_nr_pair(const float* rl, const float* nzw, int Z, float& acc0, float& acc1) {
    acc0 = 0.f;
    acc1 = 0.f;
    for (int z = 0; z < Z; ++z) {
        const float r = rl[z];
        acc0 = fmaf(nzw[z], r, acc0);
        acc1 = fmaf(nzw[Z + z], r, acc1);
    }
}

}  // namespace mpv
