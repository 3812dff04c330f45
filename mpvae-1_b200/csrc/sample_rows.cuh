// The warp and grid layout of the sampled-prediction row passes (predict.cu, sets.cu): a warp per (batch row, 128-label
// chunk), four labels per lane, the S sample rows of nr streamed through registers.
#pragma once
#include "common.cuh"
#include "rows.h"
#include "small_rows.cuh"   // row_of

namespace mpv {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kChunk = 128;   // labels per warp and iteration: four per lane, one 16-byte load per sample row
constexpr int kLL = 4;

// The S sample rows of nr at (row b, labels l0 .. l0+3), in sample order: body(s0, v) once per pair (s0, s0 + 1), with
// v[i][j] = nr[sample s0 + i, row b, label l0 + j], while the loads of the next two pairs are in flight.  Rows are
// 16-byte aligned (ldn % 4 == 0) and l0 is a multiple of 4; the pitch padding [L, ldn) is loaded but never stored.
// Past S, and everywhere when !active, v is zeros and nothing is loaded.  The scalars are taken by reference: by value,
// nvcc 12.9 schedules the callers' index arithmetic differently (one more uniform add, two registers fewer in pass A).
template <class Body>
__device__ __forceinline__ void for_sample_pairs(const RowArgs& a, const int& S, const int& b, const int& l0,
                                                 const bool& active, Body body) {
    const float* __restrict__ col = a.nr + l0;
    auto load = [&](int s) {
        float4 n = make_float4(0.f, 0.f, 0.f, 0.f);
        if (s < S && active) n = __ldcs(reinterpret_cast<const float4*>(col + row_of(a, s, b) * a.ldn));
        return n;
    };
    float4 q0 = load(0), q1 = load(1), q2 = load(2), q3 = load(3);
    for (int s0 = 0; s0 < S; s0 += 2) {
        const float4 n0 = q0, n1 = q1;
        q0 = q2; q1 = q3;
        q2 = load(s0 + 4); q3 = load(s0 + 5);
        const float v[2][kLL] = {{n0.x, n0.y, n0.z, n0.w}, {n1.x, n1.y, n1.z, n1.w}};
        body(s0, v);
    }
}

// Grid (B, G) of the row passes, a warp per 128-label chunk: the chunks of a row are dealt out to G CTAs so that the
// grid fills the GPU whatever B is -- ~2 waves of 4 resident CTAs per SM, at most one CTA per 8 chunks
dim3 rows_grid(const RowArgs& a, int nchunks) {
    int gy = ceil_div(2 * 4 * kNumSMs, a.B);
    if (gy > ceil_div(nchunks, kWarps)) gy = ceil_div(nchunks, kWarps);
    if (gy < 1) gy = 1;
    return dim3(a.B, gy);
}

}  // namespace

}  // namespace mpv
