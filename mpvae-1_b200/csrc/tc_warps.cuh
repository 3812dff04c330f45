// The roles the tcgen05 product kernel (contract_tc.cu) gives its warps beyond the TMA / MMA / promotion pipeline:
//   - the eight "math" warps of the nt product (MATH == 2) draw the Philox noise of the A operand just ahead of the tiles
//     that read it;
//   - in the g_R product of a data-parallel run (MATH == 4) a control thread publishes every finished tile in a per-tile
//     counter in peer memory, for the exchange kernel that runs beside the product (peer_reduce.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cuda_fp16.h>

#include "common.cuh"
#include "philox.cuh"

namespace mpv {

constexpr int kFuseMathWarps = 8;          // per CTA: two warpgroups

// Flag polling.  An acquire LOAD compiles to LDG.STRONG + CCTL.IVALL (an L1 invalidation) on every poll, and a few
// hundred spinning warps doing that starve the whole SM (measured: the g_R product went from 0.44 to 0.65 ms).  So the
// polls are RELAXED loads and one acquire FENCE follows the successful one.
__device__ __forceinline__ unsigned int ld_relaxed_gpu(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fence_acquire_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void fence_acquire_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ noise just in time
// The math warps' job (it pays: pure integer / SFU work with plenty of independent instructions per warp): DRAWING the
// Philox normals of mpvae.py:162 straight into the product's own A operand plane while the tensor pipe works on earlier
// rows.  The plane is cut into blocks of 128 rows (one CTA's share of a tile); all math warps of the grid fill block 0,
// then block 1, ... in the order the tiles consume them, bump the block's counter when their share is written, and the
// TMA producer of a CTA waits for its block's counter before the first load of a tile.  Same counter -> element mapping
// as philox_planes_kernel, so the numbers are identical.
struct FuseNoise {
    __half* plane;                 // [S*B][pitch] halves, rows b-major (b * S + s)
    int S, B, Z, pitch, Bg, row0;  // Bg / row0: the global batch this shard's rows [row0, row0 + B) belong to
    uint2 key, off;
    const unsigned long long* off_dev;
    unsigned int* ready;           // [ceil(S*B / 128)] counters, zeroed before the launch
};

__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// TMA producer thread: block `u` of the plane is complete once every math warp of the grid has signalled it
__device__ __forceinline__ void noise_wait_block(const unsigned int* cnt, unsigned int warps_total) {
    const long long t0 = clock64();
    while (ld_relaxed_gpu(cnt) < warps_total) {
        __nanosleep(100);
        if (clock64() - t0 > 8000000000LL) __trap();   // ~4 s: a protocol bug must not hang the GPU
    }
    fence_acquire_gpu();
    fence_proxy_async_global();                         // generic-proxy stores -> async-proxy (TMA) loads
}

// One math warp's share of the whole plane.  gw = this warp's index among the `warps_total` math warps of the grid.
__device__ __forceinline__ void noise_math_loop(const FuseNoise& f, int gw, int warps_total, int lane) {
    const int M = f.S * f.B;
    const int nblocks = (M + 127) >> 7;
    const unsigned cpr = (unsigned)((f.Z + 3) / 4 + 1);           // counters that can touch one row
    const unsigned units = 128u * cpr;
    const unsigned stride = (unsigned)warps_total * 32u;
    const uint2 off = philox_offset(f.off, f.off_dev);
    for (int u = 0; u < nblocks; ++u) {
        for (unsigned idx = (unsigned)gw * 32u + (unsigned)lane; idx < units; idx += stride) {
            const int m = (u << 7) + (int)(idx / cpr);
            if (m >= M) break;
            const int b = m / f.S, s = m - b * f.S;
            const unsigned long long flat0 = ((unsigned long long)s * f.Bg + f.row0 + b) * f.Z;   // (s, b_global, 0)
            const unsigned long long c = (flat0 >> 2) + (idx % cpr);
            const long long z0 = (long long)(c << 2) - (long long)flat0;                        // -3 .. Z + 3
            if (z0 >= f.Z) continue;
            float n[4];
            philox_normal4(c, f.key, off, n);
            __half* __restrict__ row = f.plane + (size_t)m * f.pitch;
            if (z0 >= 0 && z0 + 4 <= f.Z) {
                __half* dst = row + z0;
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
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const long long z = z0 + j;
                    if (z >= 0 && z < f.Z) row[z] = __float2half_rn(n[j]);
                }
            }
        }
        fence_proxy_async_global();
        __threadfence();
        __syncwarp();
        if (lane == 0) atomicAdd(f.ready + u, 1u);
    }
}

// ------------------------------------------------------------------------------------------------ tile publisher
// In the BACKWARD product g_R = gxs^T . noise of a data-parallel run, every rank's product writes its partial g_R into
// its own peer-mapped buffer and bumps a per-tile counter (in peer memory too) when a tile is stored; the exchange kernel
// beside it (peer_reduce.cu) sums each 256-row slab over the ranks as soon as the slab is complete on every rank.
// Counters are monotonic (a tile is complete when its counter reaches 32 x the exchange's epoch), so nothing is reset
// between steps.  The K-sliced tail wave of the product (finished by tail_fixup_kernel after this kernel) is exchanged
// afterwards by the stand-alone reduce kernel over that row range.
struct FusePeer {
    int world;                         // ranks of the run (the SMs left to the exchange: exchange_sms(world))
    unsigned int* done;                // this rank's per-tile counters
    int full_tiles;                    // tiles [0, full_tiles) are published (filled in by the launcher)
};

// Publishing a finished tile.  A system-scope fence in each of the 512 promotion threads (MEMBAR.SC.SYS + an L1
// invalidation) stalls the warps the tensor pipe is waiting for, so the promotion warps only count themselves in shared
// memory (CTA-scope release) and ONE otherwise idle control thread per CTA turns sixteen arrivals into one system-scope
// release and one bump of the tile's counter by 16 (release / acquire chains are cumulative).
__device__ __forceinline__ void peer_arrive_tile(volatile int* arrivals, int lane) {
    __threadfence_block();
    __syncwarp();
    if (lane == 0) atomicAdd_block(const_cast<int*>(arrivals), 1);
}
// control warp 3, one thread: the n-th exchangeable tile of this CTA is `t`
__device__ __forceinline__ void peer_publish_tile(const FusePeer& f, volatile int* arrivals, int n, int t) {
    while (*arrivals < 16 * (n + 1)) __nanosleep(100);
    fence_acquire_sys();                                  // acq_rel: the promotion warps' stores, then the counter
    atomicAdd(f.done + t, 16u);
}

}  // namespace mpv
