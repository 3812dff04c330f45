// Mode prediction: the model's probability of whole label sets, and per row the set that maximises it.
//
// After predict's nt product (nr in the workspace), sample s of row b has x_sl = nr[s, b, l] + fx_out[b, l], and given
// the noise the labels are independent Bernoulli(E_sl).  With the loss's fp32 cell logs (cell_forward's ll, either CDF
// mode) ll+_sl = log E_sl and ll-_sl = log(1 - E_sl):
//   A_s = sum_l ll-_sl,  d_sl = ll+_sl - ll-_sl       (fp64; the difference of two fp32 logs in [-15, 0] is exact)
//   lp_s(y) = A_s + sum_{l in y} d_sl
//   log P(y) = M + log((1 / S) sum_s exp(lp_s - M)),  M = max_s lp_s;   ess(y) = (sum_s w_s)^2 / sum_s w_s^2,
//   w_s = exp(lp_s - M)
// P is the S-component mixture predict averages, with the Bernoulli draw integrated out.
//
// Launches after the product:
//   rows     probit_mode_rows_kernel   grid and warps of probit_predict_rows_kernel: per (s, b, 128-label chunk) the
//                                      fp64 partial of A_s, d_sl for every cell, and for the mode the candidate bits
//   score    mode_score_kernel         one CTA per row: A_s (the chunk partials in chunk order), then per set lp_s (a
//                                      thread per sample up to 128 labels, else a warp per sample, lane-strided words,
//                                      the butterfly) and its log P and ess
//   ascent   mode_ascent_kernel        (mode) one CTA per row: the best candidate, then steepest single-flip ascent
//   score    mode_score_kernel         (mode) the final set, so its log P and ess are score_sets' bits
// Candidates (mode): c0 = 1[indiv_prob >= 1/2] (predict's pair sums, evals' threshold), c1 = the empty set, c_{2+s} =
// the component modes 1[ll+_s > ll-_s].  A candidate equal to an earlier one takes its score without rescoring.
// Sets are (B, C, W) int32 words in sample_labels' layout (label l at bit l % 32 of word l / 32); the bits at and
// above L are masked off at every read.
#include "../../include/mpvae_b200.h"
#include "common.cuh"
#include "probit_math.cuh"
#include "rows.h"
#include "sample_rows.cuh"   // kThreads, kChunk, kLL, for_sample_pairs, rows_grid

namespace mpv {

namespace {

constexpr int kRowThreads = 256;               // the score and ascent kernels: one CTA per row
constexpr int kRowWarps = kRowThreads / 32;

struct ModeRowArgs {
    double* part;      // (B, S, nchunks) fp64 partial of A_s per chunk
    double* d;         // (B, S, L)
    uint32_t* cand;    // (B, S + 2, W) candidate bits, or nullptr (score_sets)
    int W;
};

// cell_forward's ll for y = 1 and y = 0, sharing the one E
template <bool STABLE>
__device__ __forceinline__ void cell_logs(float x, float& E, float& llp, float& lln) {
    float om;
    if (STABLE) {
        probit_E_stable(x, E, om);
    } else {
        E = probit_E(x);
        om = MPV_ADD(1.0f, -E);
    }
    llp = MPV_LOG_NORMAL(E);
    lln = MPV_LOG_NORMAL(om);
}

// or of the lanes' four-bit groups into one word per 8 lanes (lanes 0, 8, 16, 24 hold the chunk's four words)
__device__ __forceinline__ uint32_t chunk_word(uint32_t m, int lane) {
    m <<= kLL * (lane & 7);
    m |= __shfl_xor_sync(0xffffffffu, m, 1);
    m |= __shfl_xor_sync(0xffffffffu, m, 2);
    m |= __shfl_xor_sync(0xffffffffu, m, 4);
    return m;
}

template <bool STABLE>
__global__ void __launch_bounds__(kThreads)
probit_mode_rows_kernel(const RowArgs a, const ModeRowArgs g, int nchunks) {
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = a.L, S = a.S, W = g.W;
    const size_t yoff = (size_t)b * L;
    const float fS = (float)S;
    uint32_t* __restrict__ cand = g.cand ? g.cand + (size_t)b * (S + 2) * W : nullptr;
    for (int c = blockIdx.y * kWarps + warp; c < nchunks; c += gridDim.y * kWarps) {
        const int l0 = c * kChunk + kLL * lane;
        const bool active = l0 < L;
        const int word = c * (kChunk / 32) + (lane >> 3);
        float fx[kLL], acc[kLL];
#pragma unroll
        for (int j = 0; j < kLL; ++j) {
            fx[j] = l0 + j < L ? a.fx_out[yoff + l0 + j] : 0.f;
            acc[j] = 0.f;
        }
        for_sample_pairs(a, S, b, l0, active, [&](int s0, const float (&v)[2][kLL]) {
            float e[2][kLL];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int s = s0 + i;
                if (s >= S) break;   // the same for the whole warp
                double an = 0.0;
                uint32_t m = 0;
                double* __restrict__ drow = g.d + ((size_t)b * S + s) * L;
#pragma unroll
                for (int j = 0; j < kLL; ++j) {
                    e[i][j] = 0.f;
                    if (l0 + j >= L) continue;
                    float llp, lln;
                    cell_logs<STABLE>(v[i][j] + fx[j], e[i][j], llp, lln);
                    an += (double)lln;
                    drow[l0 + j] = (double)llp - (double)lln;
                    m |= (uint32_t)(llp > lln) << j;
                }
                an = warp_sum(an);
                if (lane == 0) g.part[((size_t)b * S + s) * nchunks + c] = an;
                if (cand) {
                    m = chunk_word(m, lane);
                    if ((lane & 7) == 0 && word < W) cand[(size_t)(2 + s) * W + word] = m;
                }
            }
            if (cand) {
#pragma unroll
                for (int j = 0; j < kLL; ++j) {   // predict's pair sum, op for op
                    float pl = e[0][j];
                    if (s0 + 1 < S) pl += e[1][j];
                    acc[j] += pl;
                }
            }
        });
        if (cand) {
            uint32_t m = 0;
#pragma unroll
            for (int j = 0; j < kLL; ++j)
                if (l0 + j < L) m |= (uint32_t)(acc[j] / fS >= 0.5f) << j;   // evals' rule on predict's indiv_prob
            m = chunk_word(m, lane);
            if ((lane & 7) == 0 && word < W) {
                cand[word] = m;
                cand[W + word] = 0u;
            }
        }
    }
}

// ---- per-row kernels ----

// block reductions in a fixed order: each warp's butterfly, then the warps' results in warp order; every thread gets
// the result
__device__ __forceinline__ double block_sum_d(double v, double* red) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kRowWarps; ++w) s += red[w];
    __syncthreads();
    return s;
}

__device__ __forceinline__ double block_max_d(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double m = red[0];
#pragma unroll
    for (int w = 1; w < kRowWarps; ++w) m = fmax(m, red[w]);
    __syncthreads();
    return m;
}

// the largest v over the block and its index, ties to the lower index; a NaN never wins (index -1 when every v is NaN)
struct ArgMax { double v; int i; };
__device__ __forceinline__ bool beats(double v, int i, const ArgMax& o) {
    return v > o.v || (v == o.v && i >= 0 && (o.i < 0 || i < o.i));
}
__device__ __forceinline__ ArgMax block_argmax(ArgMax x, double* vred, int* ired) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double v = __shfl_xor_sync(0xffffffffu, x.v, o);
        const int i = __shfl_xor_sync(0xffffffffu, x.i, o);
        if (beats(v, i, x)) x = {v, i};
    }
    if ((threadIdx.x & 31) == 0) { vred[threadIdx.x >> 5] = x.v; ired[threadIdx.x >> 5] = x.i; }
    __syncthreads();
    ArgMax r{vred[0], ired[0]};
#pragma unroll
    for (int w = 1; w < kRowWarps; ++w)
        if (beats(vred[w], ired[w], r)) r = {vred[w], ired[w]};
    __syncthreads();
    return r;
}

// lp_s(y) = A_s + sum_{l in y} d_sl for every s.  Up to 128 labels (kThreadWords words) a thread per sample adds the
// set's d in label order; above, a warp per sample, each lane its words (stride 32) with their bits in label order,
// then the butterfly.  The order depends on L alone, so every call on a row's samples adds in the same order.
constexpr int kThreadWords = 4;
__device__ __forceinline__ void set_lp(const double* __restrict__ A, const double* __restrict__ d, const uint32_t* y,
                                       int S, int L, int W, uint32_t tail, double* __restrict__ lp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (W <= kThreadWords) {
        for (int s = threadIdx.x; s < S; s += kRowThreads) {
            const double* __restrict__ ds = d + (size_t)s * L;
            double acc = 0.0;
            for (int w = 0; w < W; ++w) {
                uint32_t u = y[w] & (w == W - 1 ? tail : 0xffffffffu);
                while (u) {
                    acc += ds[(w << 5) + __ffs(u) - 1];
                    u &= u - 1u;
                }
            }
            lp[s] = A[s] + acc;
        }
        __syncthreads();
        return;
    }
    for (int s = warp; s < S; s += kRowWarps) {
        const double* __restrict__ ds = d + (size_t)s * L;
        double acc = 0.0;
        for (int w = lane; w < W; w += 32) {
            uint32_t u = y[w] & (w == W - 1 ? tail : 0xffffffffu);
            while (u) {
                acc += ds[(w << 5) + __ffs(u) - 1];
                u &= u - 1u;
            }
        }
        acc = warp_sum(acc);
        if (lane == 0) lp[s] = A[s] + acc;
    }
    __syncthreads();
}

struct ScoreArgs {
    const double* part;      // (B, S, nchunks)
    const double* d;         // (B, S, L)
    double* A;               // (B, S)
    double* lp;              // (B, S)
    const uint32_t* bits;    // (B, C, W)
    double *log_prob, *ess;  // (B, C)
    int S, L, W, C, nchunks;
};

__global__ void __launch_bounds__(kRowThreads)
mode_score_kernel(const ScoreArgs p) {
    __shared__ double red[kRowWarps];
    __shared__ int s_dup[2];   // by candidate parity: a slot is rewritten only after every thread has read it
    const int b = blockIdx.x, tid = threadIdx.x;
    const int S = p.S, L = p.L, W = p.W, C = p.C;
    const uint32_t tail = (L & 31) ? (1u << (L & 31)) - 1u : 0xffffffffu;
    double* __restrict__ A = p.A + (size_t)b * S;
    double* __restrict__ lp = p.lp + (size_t)b * S;
    const double* __restrict__ d = p.d + (size_t)b * S * L;
    const uint32_t* __restrict__ rb = p.bits + (size_t)b * C * W;
    double* __restrict__ out_lp = p.log_prob + (size_t)b * C;
    double* __restrict__ out_ess = p.ess + (size_t)b * C;
    for (int s = tid; s < S; s += kRowThreads) {
        const double* __restrict__ q = p.part + ((size_t)b * S + s) * p.nchunks;
        double a = 0.0;
        for (int c = 0; c < p.nchunks; ++c) a += q[c];
        A[s] = a;
    }
    __syncthreads();
    for (int c = 0; c < C; ++c) {
        const uint32_t* __restrict__ y = rb + (size_t)c * W;
        // an earlier candidate with the same labels has this one's score already
        int* dup_slot = s_dup + (c & 1);
        if (tid == 0) *dup_slot = c;
        __syncthreads();
        for (int q = tid; q < c; q += kRowThreads) {
            const uint32_t* __restrict__ z = rb + (size_t)q * W;
            bool same = true;
            for (int w = 0; w < W && same; ++w) {
                const uint32_t m = w == W - 1 ? tail : 0xffffffffu;
                same = ((y[w] ^ z[w]) & m) == 0u;
            }
            if (same) { atomicMin(dup_slot, q); break; }
        }
        __syncthreads();
        const int dup = *dup_slot;
        if (dup < c) {
            if (tid == 0) { out_lp[c] = out_lp[dup]; out_ess[c] = out_ess[dup]; }
            continue;
        }
        set_lp(A, d, y, S, L, W, tail, lp);
        double m = -INFINITY;
        for (int s = tid; s < S; s += kRowThreads) m = fmax(m, lp[s]);
        m = block_max_d(m, red);
        double se = 0.0, s2 = 0.0;
        for (int s = tid; s < S; s += kRowThreads) {
            const double w = exp(lp[s] - m);
            se += w;
            s2 += w * w;
        }
        se = block_sum_d(se, red);
        s2 = block_sum_d(s2, red);
        if (tid == 0) {
            out_lp[c] = m + log(se / (double)S);
            out_ess[c] = se * se / s2;
        }
    }
}

struct AscentArgs {
    const double *A, *d;         // (B, S), (B, S, L)
    const uint32_t* cand;        // (B, C, W)
    const double* cand_lp;       // (B, C)
    double *lp, *wts;            // (B, S)
    uint32_t* yhat;              // (B, W)
    uint8_t* sets;               // (B, L)
    int32_t *size, *flips;       // (B)
    int S, L, W, C, max_flips;
};

// From the best candidate (ties to the earliest), flip the label with the largest gain while it is positive.  The gain
// of flipping l is log(G_l / T): T = sum_s w_s, G_l = sum_s w_s exp(+-d_sl) (+ to add l, - to remove it), both summed
// over the samples in order by one thread; the largest G_l wins, ties to the lower label, and is taken when G_l > T.
// lp_s follows each flip by +-d_sl.
__global__ void __launch_bounds__(kRowThreads)
mode_ascent_kernel(const AscentArgs p) {
    __shared__ double vred[kRowWarps];
    __shared__ int ired[kRowWarps];
    __shared__ double s_T;
    const int b = blockIdx.x, tid = threadIdx.x;
    const int S = p.S, L = p.L, W = p.W, C = p.C;
    const uint32_t tail = (L & 31) ? (1u << (L & 31)) - 1u : 0xffffffffu;
    const double* __restrict__ A = p.A + (size_t)b * S;
    const double* __restrict__ d = p.d + (size_t)b * S * L;
    double* lp = p.lp + (size_t)b * S;
    double* wts = p.wts + (size_t)b * S;
    uint32_t* y = p.yhat + (size_t)b * W;
    ArgMax best{-INFINITY, -1};
    for (int c = tid; c < C; c += kRowThreads) {
        const double v = p.cand_lp[(size_t)b * C + c];
        if (beats(v, c, best)) best = {v, c};
    }
    best = block_argmax(best, vred, ired);
    const uint32_t* __restrict__ start = p.cand + ((size_t)b * C + (best.i < 0 ? 0 : best.i)) * W;
    for (int w = tid; w < W; w += kRowThreads) y[w] = start[w] & (w == W - 1 ? tail : 0xffffffffu);
    __syncthreads();
    set_lp(A, d, y, S, L, W, tail, lp);
    int nflip = 0;
    while (nflip < p.max_flips) {
        double m = -INFINITY;
        for (int s = tid; s < S; s += kRowThreads) m = fmax(m, lp[s]);
        m = block_max_d(m, vred);
        for (int s = tid; s < S; s += kRowThreads) wts[s] = exp(lp[s] - m);
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
            for (int s = 0; s < S; ++s) t += wts[s];
            s_T = t;
        }
        ArgMax g{-INFINITY, -1};
        for (int l = tid; l < L; l += kRowThreads) {
            const bool on = (y[l >> 5] >> (l & 31)) & 1u;
            double G = 0.0;
            if (on) {
                for (int s = 0; s < S; ++s) G += wts[s] * exp(-d[(size_t)s * L + l]);
            } else {
                for (int s = 0; s < S; ++s) G += wts[s] * exp(d[(size_t)s * L + l]);
            }
            if (beats(G, l, g)) g = {G, l};
        }
        g = block_argmax(g, vred, ired);   // its barriers also publish s_T
        if (g.i < 0 || !(g.v > s_T)) break;
        const int l = g.i;
        const bool on = (y[l >> 5] >> (l & 31)) & 1u;
        for (int s = tid; s < S; s += kRowThreads) lp[s] += on ? -d[(size_t)s * L + l] : d[(size_t)s * L + l];
        __syncthreads();   // every thread has read y[l >> 5]
        if (tid == 0) y[l >> 5] ^= 1u << (l & 31);
        ++nflip;
        __syncthreads();
    }
    uint8_t* __restrict__ row = p.sets + (size_t)b * L;
    int n = 0;
    for (int l = tid; l < L; l += kRowThreads) {
        const uint8_t v = (y[l >> 5] >> (l & 31)) & 1u;
        row[l] = v;
        n += v;
    }
    n = (int)block_sum_d((double)n, vred);
    if (tid == 0) {
        p.size[b] = n;
        p.flips[b] = nflip;
    }
}

int launch_mode_rows(const RowArgs& a, const ModeLayout& w, char* base, bool candidates, cudaStream_t stream) {
    const int nchunks = (a.L + kChunk - 1) / kChunk;
    const dim3 grid = rows_grid(a, nchunks);
    ModeRowArgs g{};
    g.part = reinterpret_cast<double*>(base + w.part);
    g.d = reinterpret_cast<double*>(base + w.d);
    g.cand = candidates ? reinterpret_cast<uint32_t*>(base + w.cand) : nullptr;
    g.W = (a.L + 31) / 32;
    if (a.stable) probit_mode_rows_kernel<true><<<grid, kThreads, 0, stream>>>(a, g, nchunks);
    else probit_mode_rows_kernel<false><<<grid, kThreads, 0, stream>>>(a, g, nchunks);
    return check_launch("probit_mode_rows_kernel");
}

int launch_score(const RowArgs& a, const ModeLayout& w, char* base, const uint32_t* bits, int C, double* log_prob,
                 double* ess, cudaStream_t stream) {
    ScoreArgs p{};
    p.part = reinterpret_cast<const double*>(base + w.part);
    p.d = reinterpret_cast<const double*>(base + w.d);
    p.A = reinterpret_cast<double*>(base + w.a);
    p.lp = reinterpret_cast<double*>(base + w.lp);
    p.bits = bits;
    p.log_prob = log_prob; p.ess = ess;
    p.S = a.S; p.L = a.L; p.W = (a.L + 31) / 32; p.C = C;
    p.nchunks = (a.L + kChunk - 1) / kChunk;
    mode_score_kernel<<<a.B, kRowThreads, 0, stream>>>(p);
    return check_launch("mode_score_kernel");
}

}  // namespace

ModeLayout mode_layout(int S, int B, int L) {
    ModeLayout w{};
    const size_t nchunks = (size_t)(L + kChunk - 1) / kChunk, W = (size_t)(L + 31) / 32, C = (size_t)S + 2;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    w.part = take((size_t)B * S * nchunks * sizeof(double));
    w.a = take((size_t)B * S * sizeof(double));
    w.d = take((size_t)B * S * L * sizeof(double));
    w.lp = take((size_t)B * S * sizeof(double));
    w.wts = take((size_t)B * S * sizeof(double));
    w.cand = take((size_t)B * C * W * sizeof(uint32_t));
    w.cand_lp = take((size_t)B * C * sizeof(double));
    w.cand_ess = take((size_t)B * C * sizeof(double));
    w.yhat = take((size_t)B * W * sizeof(uint32_t));
    w.total = off;
    return w;
}

int launch_score_sets(RowArgs a, const int32_t* bits, int C, double* log_prob, double* ess, void* ws,
                      cudaStream_t stream) {
    const ModeLayout w = mode_layout(a.S, a.B, a.L);
    char* base = static_cast<char*>(ws);
    if (int rc = launch_mode_rows(a, w, base, false, stream)) return rc;
    return launch_score(a, w, base, reinterpret_cast<const uint32_t*>(bits), C, log_prob, ess, stream);
}

int launch_predict_mode(RowArgs a, int max_flips, uint8_t* sets, double* log_prob, double* ess, int32_t* size,
                        int32_t* flips, void* ws, cudaStream_t stream) {
    const ModeLayout w = mode_layout(a.S, a.B, a.L);
    char* base = static_cast<char*>(ws);
    const int C = a.S + 2;
    const uint32_t* cand = reinterpret_cast<const uint32_t*>(base + w.cand);
    double* cand_lp = reinterpret_cast<double*>(base + w.cand_lp);
    if (int rc = launch_mode_rows(a, w, base, true, stream)) return rc;
    if (int rc = launch_score(a, w, base, cand, C, cand_lp, reinterpret_cast<double*>(base + w.cand_ess), stream)) return rc;
    AscentArgs p{};
    p.A = reinterpret_cast<const double*>(base + w.a);
    p.d = reinterpret_cast<const double*>(base + w.d);
    p.cand = cand;
    p.cand_lp = cand_lp;
    p.lp = reinterpret_cast<double*>(base + w.lp);
    p.wts = reinterpret_cast<double*>(base + w.wts);
    p.yhat = reinterpret_cast<uint32_t*>(base + w.yhat);
    p.sets = sets; p.size = size; p.flips = flips;
    p.S = a.S; p.L = a.L; p.W = (a.L + 31) / 32; p.C = C; p.max_flips = max_flips;
    mode_ascent_kernel<<<a.B, kRowThreads, 0, stream>>>(p);
    if (int rc = check_launch("mode_ascent_kernel")) return rc;
    return launch_score(a, w, base, p.yhat, 1, log_prob, ess, stream);
}

}  // namespace mpv
