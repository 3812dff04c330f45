// Prediction-only kernels: indiv_prob[b, l] = mean_s E(nr[s, b, l] + fx_out[b, l]) (mpvae.py:170,180,203), the feature
// branch alone.  Scoring new rows needs no labels, so none of the loss forward's other work happens here: no label
// branch, no log-likelihoods, no ranking factors, no per-(row, sample) statistics, no per-row tail.
//
// The predictions are bit-equal to the indiv_prob of the loss forward by construction: E comes from the same
// probit_math.cuh functions (probit_E, or probit_E_stable under MPVAE_FLAG_STABLE_CDF), and the mean over samples is
// taken in the forward kernels' order -- pair sums E_s + E_{s+1}, pairs added in sample order, then / S.
#include "common.cuh"
#include "probit_math.cuh"
#include "rows.h"
#include "small_rows.cuh"

namespace mpv {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kChunk = 128;   // labels per warp and iteration: four per lane, one 16-byte load per sample row
constexpr int kLL = 4;

// After the nt product (nr in the workspace, either row layout).  A warp owns 128 neighbouring labels of one batch row
// and walks the S samples with the four running sums in registers; the loads of the next two sample pairs are in
// flight while a pair is computed.  Grid (B, G): the chunks of a row are dealt out to G CTAs so that the grid fills
// the GPU whatever B is.
template <bool STABLE>
__global__ void __launch_bounds__(kThreads)
probit_predict_rows_kernel(const RowArgs a, int nchunks) {
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = a.L, S = a.S;
    const size_t yoff = (size_t)b * L;
    const float fS = (float)S;
    for (int c = blockIdx.y * kWarps + warp; c < nchunks; c += gridDim.y * kWarps) {
        const int l0 = c * kChunk + kLL * lane;
        if (l0 >= L) continue;
        float fx[kLL], acc[kLL];
#pragma unroll
        for (int j = 0; j < kLL; ++j) {
            fx[j] = l0 + j < L ? a.fx_out[yoff + l0 + j] : 0.f;
            acc[j] = 0.f;
        }
        // rows are 16-byte aligned (ldn % 4 == 0) and l0 is a multiple of 4; the pitch padding [L, ldn) is loaded but
        // never stored
        const float* __restrict__ col = a.nr + l0;
        auto load = [&](int s) {
            float4 n = make_float4(0.f, 0.f, 0.f, 0.f);
            if (s < S) n = __ldcs(reinterpret_cast<const float4*>(col + row_of(a, s, b) * a.ldn));
            return n;
        };
        float4 q0 = load(0), q1 = load(1), q2 = load(2), q3 = load(3);
        for (int s0 = 0; s0 < S; s0 += 2) {
            const float4 n0 = q0, n1 = q1;
            q0 = q2; q1 = q3;
            q2 = load(s0 + 4); q3 = load(s0 + 5);
            const float v0[kLL] = {n0.x, n0.y, n0.z, n0.w}, v1[kLL] = {n1.x, n1.y, n1.z, n1.w};
            const bool two = s0 + 1 < S;
#pragma unroll
            for (int j = 0; j < kLL; ++j) {
                float pl = predict_E<STABLE>(v0[j] + fx[j]);   // mpvae.py:170,180
                if (two) pl += predict_E<STABLE>(v1[j] + fx[j]);
                acc[j] += pl;
            }
        }
#pragma unroll
        for (int j = 0; j < kLL; ++j)
            if (l0 + j < L) a.indiv_prob[yoff + l0 + j] = acc[j] / fS;   // mpvae.py:203
    }
}

// Small regime, one launch, one CTA per batch row: R staged by the TMA bulk copy, the noise of a sample pair per warp
// (Philox in registers or the caller's tensor), the warp-level FMA chain, E of the feature branch; pair sums in shared
// memory, added in pair order at the end.
template <bool STABLE>
__global__ void __launch_bounds__(kSmallThreads)
probit_small_predict_kernel(const SmallArgs p) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ __align__(8) unsigned long long s_bar;
    const RowArgs& a = p.a;
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = a.L, S = a.S, Z = p.Z;
    const int npairs = (S + 1) >> 1;
    float* Rs = reinterpret_cast<float*>(s_raw);                           // [L][Z]
    float* nz = Rs + (((size_t)L * Z + 3) & ~(size_t)3);                   // [kSmallWarps][2][Z]
    float* ps = nz + (size_t)kSmallWarps * 2 * Z;                          // [npairs][L] pair sums of E
    const bool bulk = small_r_stage<kSmallThreads>(Rs, p.r, L, Z, &s_bar);
    const int nch = (L + 31) >> 5;
    float fxv[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int l = (c << 5) + lane;
        fxv[c] = (c < nch && l < L) ? a.fx_out[(size_t)b * L + l] : 0.f;
    }
    small_r_wait(bulk, &s_bar);
    __syncthreads();
    const uint2 off = philox_offset(p.off, p.off_dev);
    float* nzw = nz + (size_t)warp * 2 * Z;
    for (int pair = warp; pair < npairs; pair += kSmallWarps) {
        const int s0 = pair << 1;
        small_noise_pair(nzw, p, s0, b, off, lane);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int l = (c << 5) + lane;
            if (c >= nch || l >= L) continue;
            float acc0, acc1;
            small_nr_pair(Rs + (size_t)l * Z, nzw, Z, acc0, acc1);
            float pl = predict_E<STABLE>(acc0 + fxv[c]);
            if (s0 + 1 < S) pl += predict_E<STABLE>(acc1 + fxv[c]);
            ps[(size_t)pair * L + l] = pl;
        }
        __syncwarp();   // nzw is rewritten by the next pair
    }
    __syncthreads();
    const float fS = (float)S;
    for (int l = tid; l < L; l += kSmallThreads) {
        float sx = 0.f;
        for (int q = 0; q < npairs; ++q) sx += ps[(size_t)q * L + l];
        a.indiv_prob[(size_t)b * L + l] = sx / fS;
    }
}

}  // namespace

int launch_predict_rows(RowArgs a, cudaStream_t stream) {
    const int nchunks = (a.L + kChunk - 1) / kChunk;
    // enough CTAs for ~2 waves of 4 resident CTAs per SM, at most one CTA per 8 chunks (a warp each)
    int gy = ceil_div(2 * 4 * kNumSMs, a.B);
    if (gy > ceil_div(nchunks, kWarps)) gy = ceil_div(nchunks, kWarps);
    if (gy < 1) gy = 1;
    if (a.stable) probit_predict_rows_kernel<true><<<dim3(a.B, gy), kThreads, 0, stream>>>(a, nchunks);
    else probit_predict_rows_kernel<false><<<dim3(a.B, gy), kThreads, 0, stream>>>(a, nchunks);
    return check_launch("probit_predict_rows_kernel");
}

int launch_small_predict(RowArgs a, const SmallNoise& n, cudaStream_t stream) {
    // no more than the loss forward's shared memory (which small_regime_fits bounds): R, the noise pairs, one branch
    const size_t smem = ((((size_t)a.L * n.Z + 3) & ~(size_t)3) + (size_t)kSmallWarps * 2 * n.Z +
                         (size_t)((a.S + 1) / 2) * a.L) * sizeof(float);
    static bool configured[kMaxDevices] = {};
    const int dev = device_slot();
    if (!configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(probit_small_predict_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(probit_small_predict_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(small predict): %s", cudaGetErrorString(e)); return 4; }
        configured[dev] = true;
    }
    const SmallArgs p = small_args(a, n);
    if (a.stable) probit_small_predict_kernel<true><<<a.B, kSmallThreads, smem, stream>>>(p);
    else probit_small_predict_kernel<false><<<a.B, kSmallThreads, smem, stream>>>(p);
    return check_launch("probit_small_predict_kernel");
}

}  // namespace mpv
