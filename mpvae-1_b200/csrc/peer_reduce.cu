// Data-parallel sum of g_R over NVLink peer memory (SURVEY.md 8e), one process per GPU on one node.  Every rank maps the
// others' buffers with CUDA IPC (mpvae_peer_alloc / mpvae_peer_open) and passes the tables in mpvae_probit_params.
//
//   product       each rank's gxs^T . noise writes its partial g_R into its OWN `part` buffer (ordinary local stores)
//   signal(0)     "my partial is complete": release-store of the step number into every rank's flag row 0
//   reduce+bcast  g_R is cut into `world` contiguous chunks; the owner of a chunk waits for the world's flags, PULLS the
//                 chunk from every rank's `part` (coalesced 16-byte NVLink loads), adds the partials in rank order (fixed
//                 order: every rank ends up with bit-identical sums, run to run) and stores the result into EVERY rank's
//                 g_R (coalesced 16-byte NVLink stores); the last CTA release-stores the step number into row 1
//   wait(1)       returns when all owners have delivered: g_R is complete on this rank
//
// Per rank and step (G ranks, n = L*Z floats): 4n(G-1)/G bytes in and the same out, at once (NVLink is full duplex),
// against 2 x 4n(G-1)/G each way in sequence for a ring all-reduce.
//
// A first version pushed the tiles from the product's epilogue straight into their owners' memory to overlap the
// transfer with the GEMM; measured on 2 x B200 that was slower than NCCL: a thread of the epilogue holds one ROW, so
// its 16-byte stores are 1 KiB apart and every one became its own NVLink packet (+0.17 ms on the 0.47 ms product).
//
// Buffers are reused every step; the step number in the flags orders the reuse: a rank starts its next product (which
// overwrites `part`) only after wait(1), i.e. after every owner has finished pulling.
#include <stdlib.h>

#include "common.cuh"
#include "rows.h"

namespace mpv {
namespace {

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// flags of one rank: [2 phases][8 source ranks] + [16] = CTA counter of the reduce kernel + [17] = error word
constexpr int kFlagWords = 32;
constexpr int kErrWord = 17;
constexpr int kReduceCtas = kNumSMs * 4;

// Spin until *p == want.  A peer that never arrives must not hang the GPU for ever, and a slow one (checkpointing,
// evaluation, a data-loader stall) must not poison every other rank's context either: after ctx.timeout_cycles the
// wait gives up WITHOUT trapping and records the failed flag in this rank's error word, which the host reads with
// mpvae_peer_error() and answers by falling back to NCCL (the sums of that step are then invalid).
__device__ __forceinline__ void wait_flag(const PeerCtx& ctx, const uint32_t* p, uint32_t want) {
    const long long t0 = clock64();
    while (ld_acquire_sys(p) != want) {
        __nanosleep(100);
        if (clock64() - t0 > ctx.timeout_cycles) {
            atomicMax(ctx.flags[ctx.rank] + kErrWord, want);
            return;
        }
    }
}
// the step number of this launch: host value plus the optional device counter (CUDA-graph replays)
__device__ __forceinline__ uint32_t step_of(const PeerCtx& ctx) { return ctx.step + (ctx.step_dev ? *ctx.step_dev : 0u); }

__global__ void peer_signal_kernel(PeerCtx ctx, int phase) {
    const int p = threadIdx.x;
    __threadfence_system();
    if (p < ctx.world) st_release_sys(ctx.flags[p] + phase * 8 + ctx.rank, step_of(ctx));
}

// the last kernel of an exchange: also advances the device-side step counter for the next replay
__global__ void peer_wait_kernel(PeerCtx ctx, int phase) {
    const int p = threadIdx.x;
    if (p < ctx.world) wait_flag(ctx, ctx.flags[ctx.rank] + phase * 8 + p, step_of(ctx));
    __syncthreads();
    if (p == 0 && ctx.step_dev) *ctx.step_dev += ctx.step_stride;
    if (p == 0 && ctx.epoch_dev) *ctx.epoch_dev += 1u;
}

template <int W, int U>   // world size; float4 groups per thread and iteration (all loads are issued before the adds)
__global__ void __launch_bounds__(256)
peer_reduce_bcast_kernel(PeerCtx ctx, size_t n) {
    if (threadIdx.x < W) wait_flag(ctx, ctx.flags[ctx.rank] + threadIdx.x, step_of(ctx));
    __syncthreads();
    // this rank's chunk, in units of float4 (the buffers come from cudaMalloc: 256-byte aligned)
    const size_t n4 = (n + 3) / 4, per = (n4 + W - 1) / W;
    const size_t lo = (size_t)ctx.rank * per, hi = min(n4, lo + per);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i0 = lo + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i0 < hi; i0 += stride * U) {
        if (i0 + (U - 1) * stride < hi && 4 * (i0 + (U - 1) * stride) + 4 <= n) {
            float4 v[U][W];
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int s = 0; s < W; ++s) v[u][s] = reinterpret_cast<const float4*>(ctx.part[s])[i0 + u * stride];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                float4 a = v[u][0];
#pragma unroll
                for (int s = 1; s < W; ++s) { a.x += v[u][s].x; a.y += v[u][s].y; a.z += v[u][s].z; a.w += v[u][s].w; }
#pragma unroll
                for (int p = 0; p < W; ++p) reinterpret_cast<float4*>(ctx.g_r[p])[i0 + u * stride] = a;
            }
            continue;
        }
        for (int u = 0; u < U; ++u) {
            const size_t i = i0 + u * stride;
            if (i >= hi) break;
            if (4 * i + 4 <= n) {
                float4 a = reinterpret_cast<const float4*>(ctx.part[0])[i];
                for (int s = 1; s < W; ++s) {
                    const float4 t = reinterpret_cast<const float4*>(ctx.part[s])[i];
                    a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
                }
                for (int p = 0; p < W; ++p) reinterpret_cast<float4*>(ctx.g_r[p])[i] = a;
                continue;
            }
            for (size_t e = 4 * i; e < n; ++e) {       // the last, partial float4 of the array
                float a = 0.0f;
                for (int s = 0; s < W; ++s) a += ctx.part[s][e];
                for (int p = 0; p < W; ++p) ctx.g_r[p][e] = a;
            }
        }
    }
    // the last CTA tells every rank that this owner's chunk is delivered
    __syncthreads();
    __shared__ bool last;
    if (threadIdx.x == 0) {
        __threadfence_system();
        uint32_t* counter = ctx.flags[ctx.rank] + 16;
        last = (atomicAdd(counter, 1u) == gridDim.x - 1);
        if (last) *counter = 0;
    }
    __syncthreads();
    if (last && threadIdx.x < W) {
        __threadfence_system();
        st_release_sys(ctx.flags[threadIdx.x] + 8 + ctx.rank, step_of(ctx));
    }
}

}  // namespace

size_t peer_flag_bytes() { return kFlagWords * sizeof(uint32_t); }
int peer_error_word() { return kErrWord; }

namespace {

// In-switch reduction (NVLS): `mc_part` / `mc_gr` are MULTICAST addresses of the ranks' part / g_R buffers.  One
// multimem.ld_reduce returns the sum of all ranks' copies of 16 bytes (added inside the NVSwitch), one multimem.st writes
// the result into every rank's g_R.  A rank receives n / G bytes instead of n (G - 1) / G and sends its broadcast once,
// but still feeds its whole copy to the switch; measured (profiles/r01_peer_allreduce.txt) it is no faster than the
// pull kernel at 2 or at 8 GPUs, so it is opt-in.  Same flag protocol.
__global__ void __launch_bounds__(256)
peer_reduce_nvls_kernel(PeerCtx ctx, const float* __restrict__ mc_part, float* __restrict__ mc_gr, size_t n) {
    if (threadIdx.x < ctx.world) wait_flag(ctx, ctx.flags[ctx.rank] + threadIdx.x, step_of(ctx));
    __syncthreads();
    const int W = ctx.world;
    const size_t n4 = (n + 3) / 4, per = (n4 + W - 1) / W, nfull = n / 4;
    const size_t lo = (size_t)ctx.rank * per, hi = min(n4, lo + per), vhi = min(hi, nfull);
    // four reductions in flight per thread: a multimem.ld_reduce travels to the switch and back
    constexpr int U = 4;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i0 = lo + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i0 < vhi; i0 += stride * U) {
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const size_t i = i0 + u * stride;
            if (i < vhi)
                asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                             : "=f"(v[u].x), "=f"(v[u].y), "=f"(v[u].z), "=f"(v[u].w)
                             : "l"(mc_part + 4 * i)
                             : "memory");
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const size_t i = i0 + u * stride;
            if (i < vhi)
                asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_gr + 4 * i), "f"(v[u].x),
                             "f"(v[u].y), "f"(v[u].z), "f"(v[u].w)
                             : "memory");
        }
    }
    if (nfull < n4 && nfull >= lo && nfull < hi && blockIdx.x == 0 && threadIdx.x == 0) {
        for (size_t e = 4 * nfull; e < n; ++e) {       // the last, partial float4: plain peer loads / stores
            float acc = 0.0f;
            for (int s = 0; s < W; ++s) acc += ctx.part[s][e];
            for (int p = 0; p < W; ++p) ctx.g_r[p][e] = acc;
        }
    }
    __syncthreads();
    __shared__ bool last;
    if (threadIdx.x == 0) {
        __threadfence_system();
        uint32_t* counter = ctx.flags[ctx.rank] + 16;
        last = (atomicAdd(counter, 1u) == gridDim.x - 1);
        if (last) *counter = 0;
    }
    __syncthreads();
    if (last && threadIdx.x < ctx.world) {
        __threadfence_system();
        st_release_sys(ctx.flags[threadIdx.x] + 8 + ctx.rank, step_of(ctx));
    }
}

}  // namespace

// ---- the exchange that runs BESIDE the g_R product (capi.cu forks a side stream for it) ----
// The product (contract_tc.cu, MATH = 4) leaves exchange_sms() SMs free and publishes every finished 256 x 256 tile in a
// per-tile counter in peer memory.  This kernel owns those SMs (one 512-thread CTA each, the shared-memory request keeps
// them apart): it walks the 256-row slabs of g_R in the order the product finishes them, waits until slab s is complete
// on EVERY rank, and does for the slab what peer_reduce_bcast_kernel does for the whole matrix (pull this rank's chunk of
// the slab from all ranks, add in rank order, store to all ranks) -- while the tensor pipes of the other SMs keep
// working on later slabs.  The product never waits for this kernel, so the two cannot deadlock whatever the
// scheduling; if the hardware ran them one after the other the result would be the same, only later.
struct SlabArgs {
    const unsigned int* done[8];   // every rank's per-tile counters
    unsigned int step;             // the tile epoch (step + *step_dev): a tile is complete when its counter has reached 32 x epoch
    const unsigned int* step_dev;
    int tiles_n, n_slabs;
    size_t slab_elems;             // 256 * Z floats: a multiple of 4, slabs are 16-byte aligned
};

template <int W>
__global__ void __launch_bounds__(512, 1)
peer_reduce_slabs_kernel(PeerCtx ctx, SlabArgs sa) {
    // 16 loads of 16 bytes in flight per thread whatever the world size (an SM moves what it has in flight per NVLink
    // round trip: 512 threads x 256 B = 128 KiB per ~2.5 us = ~50 GB/s per SM)
    constexpr int U = (16 / W) < 1 ? 1 : (16 / W);
    const unsigned int epoch = sa.step + (sa.step_dev ? *sa.step_dev : 0u);
    const unsigned int target = 32u * epoch;
    const size_t n4 = sa.slab_elems / 4, per = (n4 + W - 1) / W;
    const size_t lo = (size_t)ctx.rank * per, hi = min(n4, lo + per);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (int s = 0; s < sa.n_slabs; ++s) {
        if (threadIdx.x < 32) {
            // lane = tile of the slab (tiles_n <= 32); every rank's counter of that tile
            const long long t0 = clock64();
            bool ok = false;
            while (!ok) {
                ok = true;
                if ((int)threadIdx.x < sa.tiles_n)
                    for (int r = 0; r < W; ++r) {
                        unsigned int v;
                        asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(sa.done[r] + s * sa.tiles_n + threadIdx.x) : "memory");
                        ok = ok && (int)(v - target) >= 0;
                    }
                ok = __all_sync(0xffffffffu, ok);
                if (!ok) {
                    __nanosleep(500);
                    if (clock64() - t0 > ctx.timeout_cycles) { if (threadIdx.x == 0) atomicMax(ctx.flags[ctx.rank] + kErrWord, epoch); break; }
                }
            }
            asm volatile("fence.acq_rel.sys;" ::: "memory");
        }
        __syncthreads();
        const size_t base4 = (size_t)s * n4;
        for (size_t i0 = lo + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i0 < hi; i0 += stride * U) {
            float4 v[U][W];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const size_t i = i0 + u * stride;
#pragma unroll
                for (int r = 0; r < W; ++r)
                    v[u][r] = i < hi ? reinterpret_cast<const float4*>(ctx.part[r])[base4 + i] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const size_t i = i0 + u * stride;
                if (i >= hi) continue;
                float4 a = v[u][0];
#pragma unroll
                for (int r = 1; r < W; ++r) { a.x += v[u][r].x; a.y += v[u][r].y; a.z += v[u][r].z; a.w += v[u][r].w; }
#pragma unroll
                for (int r = 0; r < W; ++r) reinterpret_cast<float4*>(ctx.g_r[r])[base4 + i] = a;
            }
        }
        __syncthreads();
    }
    __threadfence_system();
}

int launch_peer_reduce_slabs(const PeerCtx& ctx, void* const* tile_done, int tiles_n, int n_slabs, size_t slab_elems, int ctas,
                             cudaStream_t stream) {
    if (n_slabs <= 0) return 0;
    if (tiles_n > 32 || (slab_elems & 3) != 0) { set_error("peer slabs: tiles_n %d / slab of %zu floats unsupported", tiles_n, slab_elems); return 1; }
    SlabArgs sa{};
    for (int i = 0; i < ctx.world; ++i) sa.done[i] = static_cast<const unsigned int*>(tile_done[i]);
    sa.step = ctx.step; sa.step_dev = ctx.step_dev;
    sa.tiles_n = tiles_n; sa.n_slabs = n_slabs; sa.slab_elems = slab_elems;
    // 160 KiB of (unused) dynamic shared memory per CTA: one CTA per SM, so `ctas` CTAs take exactly `ctas` SMs
    const size_t smem = 160 * 1024;
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
#define MPV_SLABS(Wn)                                                                                                             \
    case Wn:                                                                                                                      \
        if (!configured[dev] && cudaFuncSetAttribute(peer_reduce_slabs_kernel<Wn>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { \
            set_error("cudaFuncSetAttribute(peer slabs) failed");                                                                 \
            return 4;                                                                                                             \
        }                                                                                                                         \
        configured[dev] = true;                                                                                                   \
        peer_reduce_slabs_kernel<Wn><<<ctas, 512, smem, stream>>>(ctx, sa);                                                      \
        break;
    switch (ctx.world) {
        MPV_SLABS(2) MPV_SLABS(3) MPV_SLABS(4) MPV_SLABS(5) MPV_SLABS(6) MPV_SLABS(7) MPV_SLABS(8)
        default: set_error("peer reduce: world size %d not in [2, 8]", ctx.world); return 1;
    }
#undef MPV_SLABS
    return check_launch("peer_reduce_slabs_kernel");
}

template <int W>
static void launch_reduce_w(const PeerCtx& ctx, size_t n, int ctas, int unroll, cudaStream_t stream) {
    if (unroll >= 4 && W <= 4) peer_reduce_bcast_kernel<W, 4><<<ctas, 256, 0, stream>>>(ctx, n);
    else if (unroll >= 2) peer_reduce_bcast_kernel<W, 2><<<ctas, 256, 0, stream>>>(ctx, n);
    else peer_reduce_bcast_kernel<W, 1><<<ctas, 256, 0, stream>>>(ctx, n);
}

int launch_peer_reduce(const PeerCtx& ctx_in, size_t n, cudaStream_t stream, size_t first) {
    // [first, first + n): a sub-range of the buffers (the rows the slab exchange left over); n == 0 still runs the two
    // flag phases, which is what tells every rank that all deliveries of this step are done
    PeerCtx ctx = ctx_in;
    for (int i = 0; i < ctx.world; ++i) { ctx.part[i] += first; ctx.g_r[i] += first; }
    static const int ctas = getenv("MPVAE_PEER_CTAS") ? atoi(getenv("MPVAE_PEER_CTAS")) : kReduceCtas;
    static const int unroll = getenv("MPVAE_PEER_UNROLL") ? atoi(getenv("MPVAE_PEER_UNROLL")) : 2;
    peer_signal_kernel<<<1, 32, 0, stream>>>(ctx, 0);
    if (int rc = check_launch("peer_signal_kernel")) return rc;
    switch (ctx.world) {
        case 2: launch_reduce_w<2>(ctx, n, ctas, unroll, stream); break;
        case 3: launch_reduce_w<3>(ctx, n, ctas, unroll, stream); break;
        case 4: launch_reduce_w<4>(ctx, n, ctas, unroll, stream); break;
        case 5: launch_reduce_w<5>(ctx, n, ctas, unroll, stream); break;
        case 6: launch_reduce_w<6>(ctx, n, ctas, unroll, stream); break;
        case 7: launch_reduce_w<7>(ctx, n, ctas, unroll, stream); break;
        case 8: launch_reduce_w<8>(ctx, n, ctas, unroll, stream); break;
        default: set_error("peer reduce: world size %d not in [2, 8]", ctx.world); return 1;
    }
    if (int rc = check_launch("peer_reduce_bcast_kernel")) return rc;
    peer_wait_kernel<<<1, 32, 0, stream>>>(ctx, 1);
    return check_launch("peer_wait_kernel");
}

int launch_peer_reduce_nvls(const PeerCtx& ctx, const float* mc_part, float* mc_gr, size_t n, cudaStream_t stream) {
    if (ctx.world < 2 || ctx.world > 8) { set_error("peer reduce: world size %d not in [2, 8]", ctx.world); return 1; }
    peer_signal_kernel<<<1, 32, 0, stream>>>(ctx, 0);
    if (int rc = check_launch("peer_signal_kernel")) return rc;
    peer_reduce_nvls_kernel<<<kReduceCtas, 256, 0, stream>>>(ctx, mc_part, mc_gr, n);
    if (int rc = check_launch("peer_reduce_nvls_kernel")) return rc;
    peer_wait_kernel<<<1, 32, 0, stream>>>(ctx, 1);
    return check_launch("peer_wait_kernel");
}

}  // namespace mpv
