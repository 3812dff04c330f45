// Set prediction: joint label samples of the probit predictive distribution, and the set that maximises the expected
// F-measure over them.
//
// Sampler, after predict's nt product (nr in the workspace): per cell, E = predict_E(nr + fx_out), the E predict averages,
// and y = (U < E).  U is the caller's (S, B, L) fp32 tensor, or a Philox stream with its own key (the seed xor-ed with
// kSetKey, as conditional_ghk.cu separates its draws): one philox4x32_10 call per lane and sample serves the lane's four
// labels, counter (s * B_global + row0 + b) * ceil(L / 4) + l / 4, and U_j = (k_j + 1/2) 2^-24 with k_j = r_j >> 8.  That
// U is a 25-bit binary fraction, one bit more than fp32 carries, so U < E is decided exactly as the integer comparison
// 2 k + 1 < ceil(2^25 E) (2^25 E is exact in fp32).  Bits: (B, S, W) int32 words, W = ceil(L / 32), label l of sample s
// at bit l % 32 of word l / 32, bits at and above L zero.  Layout and grid are probit_predict_rows_kernel's.
//
// Decoder (GFM, Dembczynski et al., NIPS 2011), one CTA per row on any bits of that layout (bits at and above L are
// ignored, whatever they hold).  With s_i = popc(y_i):
//   P0 = #{i : s_i = 0} / S,  U_b = the labels set in at least one sample (ascending)
//   Delta_{l,k} = (1/S) sum_i y_{i,l} (1 + beta^2) / (beta^2 s_i + k)        (fp64, samples added in order)
//   EF(k) = the sum of the k largest Delta_{., k} over U_b, k = 1 .. min(|U_b|, max_size);  EF(0) = P0
//   k* = the smallest argmax; the set = the top k* labels of Delta_{., k*}, ties to the lower label index.
// The k-th largest Delta is found by a radix select on the fp64 bit patterns (every Delta over U_b is positive, so the
// patterns order as the values): 8 passes of 8 bits, a 256-bin shared histogram per pass.
#include "../../include/mpvae_b200.h"
#include "common.cuh"
#include "philox.cuh"
#include "probit_math.cuh"
#include "rows.h"
#include "sample_rows.cuh"   // kThreads, kChunk, kLL, for_sample_pairs, rows_grid

namespace mpv {

namespace {

constexpr uint32_t kSetKey = 0x53455421u;   // xor-ed into the Philox key: a stream disjoint from the noise and GHK's

struct SampleArgs {
    const float* uniform;   // (S, B, L) or nullptr
    uint32_t* bits;         // (B, S, W)
    int W, quads;           // quads = ceil(L / 4): Philox counters per (sample, row)
    int Bg, row0;
    uint2 key, off;
    const unsigned long long* off_dev;
};

// bit j = y of label l0 + j of sample s (labels at and above L give 0)
template <bool STABLE>
__device__ __forceinline__ uint32_t lane_bits(const RowArgs& a, const SampleArgs& g, int s, int b, int l0,
                                              const float (&v)[kLL], const float (&fx)[kLL], uint2 off) {
    uint32_t m = 0;
    if (g.uniform) {
        const float* __restrict__ u = g.uniform + ((size_t)s * a.B + b) * a.L + l0;
#pragma unroll
        for (int j = 0; j < kLL; ++j)
            if (l0 + j < a.L) m |= (uint32_t)(__ldcs(u + j) < predict_E<STABLE>(v[j] + fx[j])) << j;
        return m;
    }
    const unsigned long long c =
        ((unsigned long long)s * g.Bg + (unsigned long long)(g.row0 + b)) * (unsigned long long)g.quads + (l0 >> 2);
    const uint4 r = philox4x32_10(make_uint4((uint32_t)c, (uint32_t)(c >> 32), off.x, off.y), g.key);
    const uint32_t rr[kLL] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int j = 0; j < kLL; ++j) {
        if (l0 + j >= a.L) continue;
        const int y2 = __float2int_ru(predict_E<STABLE>(v[j] + fx[j]) * 33554432.0f);   // ceil(2^25 E)
        m |= (uint32_t)((int)(2u * (rr[j] >> 8) + 1u) < y2) << j;
    }
    return m;
}

// A warp owns 128 neighbouring labels of one batch row and walks the S samples; per sample, the lanes' four-bit groups
// are or-ed into one word per 8 lanes, and lanes 0, 8, 16, 24 store the chunk's four words.
template <bool STABLE>
__global__ void __launch_bounds__(kThreads)
probit_sample_labels_kernel(const RowArgs a, const SampleArgs g, int nchunks) {
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = a.L, S = a.S;
    const size_t yoff = (size_t)b * L;
    const uint2 off = philox_offset(g.off, g.off_dev);
    uint32_t* __restrict__ out = g.bits + (size_t)b * S * g.W;
    for (int c = blockIdx.y * kWarps + warp; c < nchunks; c += gridDim.y * kWarps) {
        const int l0 = c * kChunk + kLL * lane;
        const bool active = l0 < L;
        const int word = c * (kChunk / 32) + (lane >> 3);
        float fx[kLL];
#pragma unroll
        for (int j = 0; j < kLL; ++j) fx[j] = l0 + j < L ? a.fx_out[yoff + l0 + j] : 0.f;
        for_sample_pairs(a, S, b, l0, active, [&](int s0, const float (&v)[2][kLL]) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int s = s0 + i;
                if (s >= S) break;   // the same for the whole warp
                uint32_t m = active ? lane_bits<STABLE>(a, g, s, b, l0, v[i], fx, off) << (kLL * (lane & 7)) : 0u;
                m |= __shfl_xor_sync(0xffffffffu, m, 1);
                m |= __shfl_xor_sync(0xffffffffu, m, 2);
                m |= __shfl_xor_sync(0xffffffffu, m, 4);
                if ((lane & 7) == 0 && word < g.W) out[(size_t)s * g.W + word] = m;
            }
        });
    }
}

// ---- decoder ----

constexpr int kDecThreads = 256;
constexpr int kDecWarps = kDecThreads / 32;

struct DecArgs {
    const uint32_t* bits;   // (B, S, W)
    int S, L, W, max_size;
    double beta2;
    uint8_t* sets;          // (B, L)
    double* expected_f;     // (B)
    int32_t* set_size;      // (B)
    int* card;              // (B, S) s_i
    double* wsmp;           // (B, S) (1 + beta^2) / (beta^2 s_i + k) of the current k
    int* ulist;             // (B, L) U_b in ascending order
    double* delta;          // (B, L) Delta_{u, k} at U_b's positions
};

// block sums in a fixed order: each warp's butterfly, then the warps' sums in warp order; every thread gets the result
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* red) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    T s = 0;
#pragma unroll
    for (int w = 0; w < kDecWarps; ++w) s += red[w];
    __syncthreads();
    return s;
}

struct Select { unsigned long long t; int ties; };   // the k-th largest's bits, and how many copies of it the top k hold

// the k-th largest of delta[0 .. n) (all positive), by 8-bit radix passes from the top byte down
__device__ Select radix_select(const double* __restrict__ delta, int n, int k, unsigned int* hist, unsigned long long* sh) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned long long prefix = 0, pmask = 0;
    int want = k;
    for (int shift = 56; shift >= 0; shift -= 8) {
        hist[tid] = 0;   // kDecThreads == 256 bins
        __syncthreads();
        for (int p = tid; p < n; p += kDecThreads) {
            const unsigned long long x = (unsigned long long)__double_as_longlong(delta[p]);
            if ((x & pmask) == prefix) atomicAdd(&hist[(x >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (warp == 0) {
            // lane i holds bins 255 - 8i down to 248 - 8i; find the bin where the running count from the top reaches want
            int cnt[8], tot = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) { cnt[q] = (int)hist[255 - 8 * lane - q]; tot += cnt[q]; }
            int inc = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            const unsigned hit = __ballot_sync(0xffffffffu, inc >= want);
            const int first = __ffs(hit) - 1;
            if (lane == first) {
                int run = inc - tot, pick = 7;
                bool found = false;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    if (found) continue;
                    if (run + cnt[q] >= want) { pick = q; found = true; }
                    else run += cnt[q];
                }
                sh[0] = prefix | ((unsigned long long)(255 - 8 * lane - pick) << shift);
                sh[1] = (unsigned long long)(want - run);
            }
        }
        __syncthreads();
        prefix = sh[0];
        want = (int)sh[1];
        pmask |= 255ull << shift;
        __syncthreads();
    }
    return {prefix, want};
}

// Delta_{u, k} for every u of U_b (a thread per label, samples in order), after the per-sample weights of k
__device__ void fill_delta(const DecArgs& d, const uint32_t* __restrict__ rb, const int* __restrict__ card,
                           double* __restrict__ wsmp, const int* __restrict__ ulist, double* __restrict__ delta, int nu,
                           int k) {
    const double num = 1.0 + d.beta2;
    for (int s = threadIdx.x; s < d.S; s += kDecThreads) wsmp[s] = num / (d.beta2 * (double)card[s] + (double)k);
    __syncthreads();
    for (int p = threadIdx.x; p < nu; p += kDecThreads) {
        const int l = ulist[p];
        const uint32_t* __restrict__ col = rb + (l >> 5);
        const int bit = l & 31;
        double acc = 0.0;
        for (int s = 0; s < d.S; ++s)
            if ((__ldg(col + (size_t)s * d.W) >> bit) & 1u) acc += wsmp[s];
        delta[p] = acc / (double)d.S;
    }
    __syncthreads();
}

// EF(k) = the sum of the k largest Delta: the ones above the k-th largest t, then the ties' copies of t
__device__ double topk_sum(const double* __restrict__ delta, int nu, const Select& sel, double* red) {
    double s = 0.0;
    for (int p = threadIdx.x; p < nu; p += kDecThreads)
        if ((unsigned long long)__double_as_longlong(delta[p]) > sel.t) s += delta[p];
    return block_sum(s, red) + (double)sel.ties * __longlong_as_double((long long)sel.t);
}

__global__ void __launch_bounds__(kDecThreads)
f1_sets_kernel(const DecArgs d) {
    __shared__ unsigned int hist[256];
    __shared__ unsigned long long sh[2];
    __shared__ double dred[kDecWarps];
    __shared__ int ired[kDecWarps];
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int S = d.S, L = d.L, W = d.W;
    const uint32_t* __restrict__ rb = d.bits + (size_t)b * S * W;
    int* __restrict__ card = d.card + (size_t)b * S;
    double* __restrict__ wsmp = d.wsmp + (size_t)b * S;
    int* __restrict__ ulist = d.ulist + (size_t)b * L;
    double* __restrict__ delta = d.delta + (size_t)b * L;
    // the bits at and above L in the last word are not labels: whatever a caller left there is masked off at every
    // read, so s_i, U_b (and through it ulist, delta and the set) only ever see labels [0, L)
    const uint32_t tail = (L & 31) ? (1u << (L & 31)) - 1u : 0xffffffffu;
    auto word = [&](int s, int w) { return __ldg(rb + (size_t)s * W + w) & (w == W - 1 ? tail : 0xffffffffu); };
    // s_i, a warp per sample, and the empty samples
    int zeros = 0;
    for (int s = warp; s < S; s += kDecWarps) {
        int c = 0;
        for (int w = lane; w < W; w += 32) c += __popc(word(s, w));
        c = warp_sum(c);
        if (lane == 0) { card[s] = c; zeros += c == 0; }
    }
    zeros = block_sum(zeros, ired);
    // U_b: the or of the samples' words, compacted in label order (256 words per round, a block-wide exclusive scan)
    int nu = 0;
    for (int w0 = 0; w0 < W; w0 += kDecThreads) {
        const int w = w0 + tid;
        uint32_t u = 0;
        if (w < W)
            for (int s = 0; s < S; ++s) u |= word(s, w);
        const int n = __popc(u);
        int inc = n;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) ired[warp] = inc;
        __syncthreads();
        int base = nu;
        for (int q = 0; q < warp; ++q) base += ired[q];
        int total = 0;
#pragma unroll
        for (int q = 0; q < kDecWarps; ++q) total += ired[q];
        int pos = base + inc - n;
        while (u) {
            const int bit = __ffs(u) - 1;
            ulist[pos++] = (w << 5) + bit;
            u &= u - 1u;
        }
        nu += total;
        __syncthreads();
    }
    // EF(k) for k = 1 .. min(|U_b|, max_size); the smallest argmax, EF(0) = P0 included
    double best = (double)zeros / (double)S;
    int kbest = 0;
    const int K = min(nu, d.max_size);
    for (int k = 1; k <= K; ++k) {
        fill_delta(d, rb, card, wsmp, ulist, delta, nu, k);
        const Select sel = radix_select(delta, nu, k, hist, sh);
        const double ef = topk_sum(delta, nu, sel, dred);
        if (ef > best) { best = ef; kbest = k; }
    }
    // the set: the top k* labels of Delta_{., k*}, ties to the lower label index
    uint8_t* __restrict__ row = d.sets + (size_t)b * L;
    for (int l = tid; l < L; l += kDecThreads) row[l] = 0;
    if (kbest > 0) {
        fill_delta(d, rb, card, wsmp, ulist, delta, nu, kbest);
        const Select sel = radix_select(delta, nu, kbest, hist, sh);
        for (int p = tid; p < nu; p += kDecThreads)
            if ((unsigned long long)__double_as_longlong(delta[p]) > sel.t) row[ulist[p]] = 1;
        if (warp == 0) {
            int seen = 0;
            for (int p0 = 0; p0 < nu && seen < sel.ties; p0 += 32) {
                const int p = p0 + lane;
                const bool tie = p < nu && (unsigned long long)__double_as_longlong(delta[p]) == sel.t;
                const unsigned bal = __ballot_sync(0xffffffffu, tie);
                if (tie && seen + __popc(bal & ((1u << lane) - 1u)) < sel.ties) row[ulist[p]] = 1;
                seen += __popc(bal);
            }
        }
    }
    if (tid == 0) {
        d.expected_f[b] = best;
        d.set_size[b] = kbest;
    }
}

}  // namespace

int launch_sample_labels(RowArgs a, const SampleInputs& in, cudaStream_t stream) {
    const int nchunks = (a.L + kChunk - 1) / kChunk;
    const dim3 grid = rows_grid(a, nchunks);
    SampleArgs g{};
    g.uniform = in.uniform;
    g.bits = reinterpret_cast<uint32_t*>(in.bits);
    g.W = (a.L + 31) / 32;
    g.quads = (a.L + 3) / 4;
    g.Bg = in.rows.b_global; g.row0 = in.rows.row0;
    g.key = make_uint2((uint32_t)in.rows.seed ^ kSetKey, (uint32_t)(in.rows.seed >> 32));
    g.off = make_uint2((uint32_t)in.rows.offset, (uint32_t)(in.rows.offset >> 32));
    g.off_dev = reinterpret_cast<const unsigned long long*>(in.rows.offset_dev);
    if (a.stable) probit_sample_labels_kernel<true><<<grid, kThreads, 0, stream>>>(a, g, nchunks);
    else probit_sample_labels_kernel<false><<<grid, kThreads, 0, stream>>>(a, g, nchunks);
    return check_launch("probit_sample_labels_kernel");
}

F1Layout f1_layout(int B, int S, int L) {
    F1Layout w{};
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    w.card = take((size_t)B * S * sizeof(int));
    w.wsmp = take((size_t)B * S * sizeof(double));
    w.ulist = take((size_t)B * L * sizeof(int));
    w.delta = take((size_t)B * L * sizeof(double));
    w.total = off;
    return w;
}

int launch_f1_sets(const int32_t* bits, int B, int S, int L, double beta, int max_size, uint8_t* sets, double* expected_f,
                   int32_t* set_size, void* ws, cudaStream_t stream) {
    const F1Layout w = f1_layout(B, S, L);
    char* base = static_cast<char*>(ws);
    DecArgs d{};
    d.bits = reinterpret_cast<const uint32_t*>(bits);
    d.S = S; d.L = L; d.W = (L + 31) / 32; d.max_size = max_size;
    d.beta2 = beta * beta;
    d.sets = sets; d.expected_f = expected_f; d.set_size = set_size;
    d.card = reinterpret_cast<int*>(base + w.card);
    d.wsmp = reinterpret_cast<double*>(base + w.wsmp);
    d.ulist = reinterpret_cast<int*>(base + w.ulist);
    d.delta = reinterpret_cast<double*>(base + w.delta);
    f1_sets_kernel<<<B, kDecThreads, 0, stream>>>(d);
    return check_launch("f1_sets_kernel");
}

}  // namespace mpv
