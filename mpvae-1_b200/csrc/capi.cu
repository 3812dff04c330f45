// extern "C" surface of libmpvae_b200 (include/mpvae_b200.h): argument validation, workspace carving and the
// launch sequence of one forward / backward of the probit ELBO.
#include <atomic>
#include <map>
#include <mutex>
#include <stdlib.h>
#include <string.h>
#include <utility>
#include <vector>

#include "../../include/mpvae_b200.h"
#include "common.cuh"
#include "rows.h"
#include "tc.h"
#include "tc_warps.cuh"

namespace mpv {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }
int check_launch(const char* what) {
    count_launch(1);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
        return 2;
    }
    return 0;
}

namespace {

// ---- per-kernel CUDA-event timing (mpvae_profile*) ----
struct ProfState {
    bool on = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pool[MPVAE_PROF_SLOTS];
    int used[MPVAE_PROF_SLOTS] = {};
};
ProfState g_prof;
std::mutex g_prof_mu;

// records an event pair around the launches issued during its lifetime (no-op unless profiling is on)
struct ProfScope {
    cudaEvent_t stop = nullptr;
    cudaStream_t stream;
    ProfScope(int slot, cudaStream_t st) : stream(st) {
        if (!g_prof.on) return;
        std::lock_guard<std::mutex> lk(g_prof_mu);
        auto& pool = g_prof.pool[slot];
        if (g_prof.used[slot] == (int)pool.size()) {
            cudaEvent_t e0, e1;
            if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return;
            pool.emplace_back(e0, e1);
        }
        auto& pr = pool[g_prof.used[slot]++];
        cudaEventRecord(pr.first, stream);
        stop = pr.second;
    }
    ~ProfScope() { if (stop) cudaEventRecord(stop, stream); }
};

// Workspace carve-up.  Everything is 256-byte aligned; the same function sizes and places.
struct Workspace {
    size_t nr, lp, stat, wts, rowaux, rowout, slots, gxs;
    size_t e_l, e_x;                              // training: clamped probabilities of both branches, kept for the backward
    size_t fuse_part;                             // forward: per-(sample-row, label chunk) partial sums
    size_t noise_f32;                             // FMA engine, library-side noise
    size_t noise_planes, r_planes, gxs_planes;    // tensor engine operand planes (noise planes persist fwd -> bwd)
    size_t fma_partials;                          // FMA engine split-K partials of g_R
    size_t small_partials;                        // small regime: per-row contributions to g_R
    size_t tn_tail;                               // tensor engine: K-slices of the g_R product's last wave
    size_t slots_bytes;                           // slots + the counters below (zeroed together at the start of a forward)
    size_t noise_counters;                        // byte offset inside the slots block
    size_t total;
};
// 32-bit slots of the first 256 bytes of the `slots` block; the counters of the just-in-time noise follow
enum { SLOT_COUNTER = 0, SLOT_ABSMAX_R = 1, SLOT_ABSMAX_GXS = 2, SLOT_ABSMAX_GP = 3 /* and 4 */, SLOT_ABSMAX_LW = 5 };

// row pitch (floats) of the (S*B, L) scratch matrices nr and gxs: 16-byte aligned rows for vector loads / stores
int row_pitch(int L) { return (L + 3) & ~3; }

bool use_tensor(uint32_t flags, int S, int B, int L, int Z) {
    if (flags & MPVAE_FLAG_CONTRACT_FMA) return false;
    if (!tc_available()) return false;
    if (Z < 8 || L < 8) return false;   // the plane writers assume at least a few elements per row
    if (flags & MPVAE_FLAG_CONTRACT_TENSOR) return true;
    // dense-GEMM regime (north star: label / rank sets >= 128)
    return Z >= 128 && L >= 128 && (long long)S * B >= 128;
}

// label / rank sets that fit an SM: one fused CTA per batch row (probit_small_fwd_kernel)
bool use_small(uint32_t flags, int S, int B, int L, int Z) {
    if (flags & (MPVAE_FLAG_CONTRACT_FMA | MPVAE_FLAG_CONTRACT_TENSOR | MPVAE_FLAG_STABLE_CDF)) return false;
    return !use_tensor(flags, S, B, L, Z) && small_regime_fits(S, B, L, Z);
}

Workspace carve(int S, int B, int L, int Z, bool want_backward, uint32_t flags) {
    Workspace w{};
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t cube = (size_t)S * B * row_pitch(L);
    const bool tensor = use_tensor(flags, S, B, L, Z);
    const int M = S * B;
    w.nr = take(cube * sizeof(float));
    w.lp = take((size_t)B * S * 2 * sizeof(double));
    w.stat = take((size_t)B * S * 4 * sizeof(float));
    w.wts = take((size_t)B * S * 2 * sizeof(float));
    w.rowaux = take((size_t)B * 2 * sizeof(float));
    w.rowout = take((size_t)B * 8 * sizeof(double));
    // [256 B of slots][per-128-row-block counters of the just-in-time noise]
    w.noise_counters = 256;
    w.slots_bytes = w.noise_counters + (tensor ? align_up((size_t)ceil_div(M, 128) * sizeof(uint32_t), 256) : 0);
    w.slots = take(w.slots_bytes);
    // everything the forward writes and the backward reads sits before the backward-only buffers, so a forward
    // sized for inference and a forward sized for training place the shared buffers identically
    w.fuse_part = take((size_t)M * row_chunks(L) * sizeof(FusePart));
    if (tensor) {
        w.noise_planes = take(tc_planes_bytes(M, Z));
        w.r_planes = take(tc_planes_bytes(L, Z));
    } else {
        w.noise_f32 = take((size_t)M * Z * sizeof(float));
    }
    if (want_backward) {
        w.e_l = take(cube * sizeof(float));
        w.e_x = take(cube * sizeof(float));
        if (tensor) {
            // the row backward writes gxs straight as operand planes (no fp32 cube, no split pass)
            w.tn_tail = take(tc_tail_scratch_bytes());
            w.gxs_planes = take(tc_planes_bytes(M, L));
        } else {
            w.gxs = take(cube * sizeof(float));
            w.fma_partials = take(contract_tn_fma_workspace(M, L, Z));
            if (use_small(flags, S, B, L, Z)) w.small_partials = take(small_partial_bytes(B, L, Z));
        }
    }
    w.total = off;
    return w;
}

// A binding that stops before the peer_* fields passes MPVAE_PARAMS_BASE_BYTES; the rest defaults to "off".
const mpvae_probit_params* normalize(const mpvae_probit_params* p, mpvae_probit_params* tmp) {
    if (p == nullptr) { set_error("params is NULL"); return nullptr; }
    if (p->struct_bytes == sizeof(mpvae_probit_params)) return p;
    if (p->struct_bytes == MPVAE_PARAMS_BASE_BYTES) {
        memset(tmp, 0, sizeof(*tmp));
        memcpy(tmp, p, MPVAE_PARAMS_BASE_BYTES);
        tmp->struct_bytes = sizeof(mpvae_probit_params);
        return tmp;
    }
    set_error("params.struct_bytes=%u, library expects %zu (or the base prefix %u) (ABI %d)", p->struct_bytes,
              sizeof(mpvae_probit_params), MPVAE_PARAMS_BASE_BYTES, MPVAE_ABI_VERSION);
    return nullptr;
}

// Rows [row0, row0 + B) must lie in the global batch that keys a Philox stream the library draws (library_draws);
// `what` names that stream in the message.
int check_rows_fit(const mpvae_probit_params* p, bool library_draws, const char* what) {
    if (library_draws && (p->noise_row0 < 0 || p->noise_b_global < p->noise_row0 + p->B)) {
        set_error("%s: rows [%d, %d) do not fit a global batch of %d", what, p->noise_row0, p->noise_row0 + p->B,
                  p->noise_b_global);
        return 1;
    }
    return 0;
}

// A scratch block an entry point takes besides the params' workspace: present, at least `need` bytes, 256-byte aligned.
// `what` names the block in the messages; `sized_for`, when not NULL, says what its size was computed for.
int check_scratch(const char* what, const void* ptr, uint64_t have, uint64_t need, const char* sized_for = nullptr) {
    if (!ptr) { set_error("NULL pointer (%s)", what); return 1; }
    if (have < need) {
        set_error("%s too small%s%s: %llu < %llu bytes", what, sized_for ? " for " : "", sized_for ? sized_for : "",
                  (unsigned long long)have, (unsigned long long)need);
        return 1;
    }
    if ((reinterpret_cast<uintptr_t>(ptr) & 255u) != 0) { set_error("%s must be 256-byte aligned", what); return 1; }
    return 0;
}

PhiloxRows philox_rows(const mpvae_probit_params* p) {
    return PhiloxRows{p->noise_b_global, p->noise_row0, p->noise_seed, p->noise_offset, p->noise_offset_dev};
}

int check_workspace(const mpvae_probit_params* p, bool backward) {
    const uint64_t need = mpvae_workspace_bytes(p->S, p->B, p->L, p->Z, backward ? 1 : 0, p->flags);
    if (p->workspace_bytes < need) {
        set_error("workspace too small: %llu < %llu bytes", (unsigned long long)p->workspace_bytes, (unsigned long long)need);
        return 1;
    }
    if ((reinterpret_cast<uintptr_t>(p->workspace) & 255u) != 0) { set_error("workspace must be 256-byte aligned"); return 1; }
    return 0;
}

int validate(const mpvae_probit_params* p, bool backward) {
    if (p->S <= 0 || p->B <= 0 || p->L <= 0 || p->Z <= 0 || p->D < 0) {
        set_error("bad sizes S=%d B=%d L=%d Z=%d D=%d (empty batches are handled by the host wrapper)", p->S, p->B, p->L,
                  p->Z, p->D);
        return 1;
    }
    if ((long long)p->S * p->B > 0x7fffffffLL) { set_error("S*B overflows int32"); return 1; }
    if (!p->y || !p->fe_out || !p->fx_out || !p->r || !p->workspace) {
        set_error("NULL input pointer (y/fe_out/fx_out/r/workspace)");
        return 1;
    }
    if (int rc = check_rows_fit(p, !p->noise, "library-side noise")) return rc;
    if (p->D > 0 && (!p->fe_mu || !p->fe_logvar || !p->fx_mu || !p->fx_logvar)) { set_error("NULL mu/logvar pointer"); return 1; }
    if (!backward && (!p->scalars[0] || !p->scalars[1] || !p->scalars[2] || !p->scalars[3] || !p->scalars[4] ||
                      !p->scalars[5] || !p->indiv_prob || !p->indiv_prob_label)) { set_error("NULL forward output pointer"); return 1; }
    if (backward) {
        if (!p->g_fe_out || !p->g_fx_out) { set_error("NULL g_fe_out/g_fx_out"); return 1; }
        if (p->D > 0 && (!p->g_fe_mu || !p->g_fe_logvar || !p->g_fx_mu || !p->g_fx_logvar)) { set_error("NULL mu/logvar gradient pointer"); return 1; }
    }
    return check_workspace(p, backward);
}

// mpvae_probit_predict reads fx_out, r, the noise fields and indiv_prob only (mpvae_probit_sample_labels: no indiv_prob)
int validate_predict(const mpvae_probit_params* p, bool writes_prob) {
    if (p->S <= 0 || p->B <= 0 || p->L <= 0 || p->Z <= 0) {
        set_error("bad sizes S=%d B=%d L=%d Z=%d (empty batches are handled by the host wrapper)", p->S, p->B, p->L, p->Z);
        return 1;
    }
    if ((long long)p->S * p->B > 0x7fffffffLL) { set_error("S*B overflows int32"); return 1; }
    if (!p->fx_out || !p->r || !p->workspace) { set_error("NULL input pointer (fx_out/r/workspace)"); return 1; }
    if (int rc = check_rows_fit(p, !p->noise, "library-side noise")) return rc;
    if (writes_prob && !p->indiv_prob) { set_error("NULL forward output pointer (indiv_prob)"); return 1; }
    return check_workspace(p, false);
}

// side stream + events of the exchange that runs beside the g_R product (one process per GPU: created once per device,
// at the first data-parallel backward -- i.e. during warm-up, never under CUDA-graph capture)
struct SideStream { cudaStream_t stream; cudaEvent_t fork, join; };
SideStream* side_stream() {
    static SideStream ss[64];
    static int state[64] = {};      // 0 = not created, 1 = ok, -1 = failed
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (state[dev] == 0) {
        state[dev] = -1;
        if (cudaStreamCreateWithFlags(&ss[dev].stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&ss[dev].fork, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&ss[dev].join, cudaEventDisableTiming) == cudaSuccess)
            state[dev] = 1;
    }
    if (state[dev] != 1) { set_error("peer: side stream unavailable"); return nullptr; }
    return &ss[dev];
}

// Exchanges that go through the per-tile counters (beside / inside the product): the counters are monotonic and a tile is
// complete when its counter has reached 32 x the epoch of the exchange.  The epoch lives on the DEVICE, in the last word
// of the rank's own counter buffer (zeroed at allocation): the kernels read 1 + that word, the last kernel of the exchange
// advances it -- so a captured CUDA graph replays correctly, and exchanges that do not touch the counters (the
// stand-alone reduce, mpvae_peer_allreduce) leave it alone.  Every rank makes the same calls, so the epochs agree.
constexpr size_t kTileEpochWord = MPVAE_PEER_TILE_BYTES / sizeof(uint32_t) - 1;

long long peer_timeout_cycles() {
    static long long v = 0;
    if (v == 0) {
        const char* e = getenv("MPVAE_PEER_TIMEOUT_S");
        double sec = e ? atof(e) : 120.0;
        if (sec < 1.0) sec = 1.0;
        v = (long long)(sec * 1.9e9);        // SM clock <= 1.965 GHz
    }
    return v;
}

RowArgs row_args(const mpvae_probit_params* p, const Workspace& w) {
    char* base = static_cast<char*>(p->workspace);
    RowArgs a{};
    a.S = p->S; a.B = p->B; a.L = p->L; a.D = p->D;
    const bool tensor = use_tensor(p->flags, p->S, p->B, p->L, p->Z);
    a.row_sb = tensor ? p->S : 1;      // b-major behind the tensor engine, s-major behind the CUDA-core contraction
    a.row_ss = tensor ? 1 : p->B;
    a.ldn = row_pitch(p->L);
    a.sanitize = (p->flags & MPVAE_FLAG_SANITIZE_DEGENERATE) ? 1 : 0;
    a.stable = (p->flags & MPVAE_FLAG_STABLE_CDF) ? 1 : 0;
    a.nll_coeff = p->nll_coeff; a.c_coeff = p->c_coeff;
    a.y = p->y; a.fe_out = p->fe_out; a.fx_out = p->fx_out;
    a.fe_mu = p->fe_mu; a.fe_logvar = p->fe_logvar; a.fx_mu = p->fx_mu; a.fx_logvar = p->fx_logvar;
    a.nr = reinterpret_cast<const float*>(base + w.nr);
    a.lp = reinterpret_cast<double*>(base + w.lp);
    a.stat = reinterpret_cast<float*>(base + w.stat);
    a.wts = reinterpret_cast<float*>(base + w.wts);
    a.rowaux = reinterpret_cast<float*>(base + w.rowaux);
    a.rowout = reinterpret_cast<double*>(base + w.rowout);
    a.counter = reinterpret_cast<unsigned int*>(base + w.slots) + SLOT_COUNTER;
    a.part = reinterpret_cast<const FusePart*>(base + w.fuse_part);
    for (int i = 0; i < 6; ++i) { a.scalars[i] = p->scalars[i]; a.g_scalars[i] = p->g_scalars[i]; }
    a.indiv_prob = p->indiv_prob; a.indiv_prob_label = p->indiv_prob_label;
    a.g_indiv_prob = p->g_indiv_prob; a.g_indiv_prob_label = p->g_indiv_prob_label;
    a.g_fe_out = p->g_fe_out; a.g_fx_out = p->g_fx_out;
    a.g_fe_mu = p->g_fe_mu; a.g_fe_logvar = p->g_fe_logvar; a.g_fx_mu = p->g_fx_mu; a.g_fx_logvar = p->g_fx_logvar;
    return a;
}

// Dense regime, up to and including the product: the noise operand (unless the product kernel draws it), the R split and
// nr = noise . R^T on tcgen05.  The caller has zeroed the slots block.
int dense_nt_product(const mpvae_probit_params* p, const Workspace& w, cudaStream_t stream) {
    char* base = static_cast<char*>(p->workspace);
    float* nr = reinterpret_cast<float*>(base + w.nr);
    uint32_t* slots = reinterpret_cast<uint32_t*>(base + w.slots);
    const int M = p->S * p->B;
    void* npl = base + w.noise_planes;
    void* rpl = base + w.r_planes;
    // library noise: drawn by the product kernel's own math warps just ahead of the tiles (unless the caller asks for
    // the separate kernel)
    const bool jit_noise = !p->noise && !(p->flags & MPVAE_FLAG_SEPARATE_NOISE);
    int rc = 0;
    if (!jit_noise) {
        ProfScope ps(MPVAE_PROF_NOISE, stream);
        // operand rows are b-major (b * S + s): the S sample-rows of a batch row are neighbours
        if (p->noise) rc = tc_split(p->noise, M, p->Z, npl, nullptr, 0, stream, 0, p->S, p->B);   // |N(0,1)| fits fp16 at scale 1
        else rc = tc_philox_planes(npl, p->S, p->B, p->Z, p->noise_b_global, p->noise_row0, p->noise_seed, p->noise_offset, p->noise_offset_dev, stream);
    }
    if (rc) return rc;
    {
        ProfScope ps(MPVAE_PROF_SPLIT_R, stream);
        rc = tc_split(p->r, p->L, p->Z, rpl, slots + SLOT_ABSMAX_R, 1, stream);
    }
    if (rc) return rc;
    FuseNoise fnz{};
    if (jit_noise) {
        fnz.plane = static_cast<__half*>(npl);
        fnz.S = p->S; fnz.B = p->B; fnz.Z = p->Z; fnz.pitch = tc_pitch(p->Z);
        fnz.Bg = p->noise_b_global; fnz.row0 = p->noise_row0;
        fnz.key = make_uint2((uint32_t)p->noise_seed, (uint32_t)(p->noise_seed >> 32));
        fnz.off = make_uint2((uint32_t)p->noise_offset, (uint32_t)(p->noise_offset >> 32));
        fnz.off_dev = reinterpret_cast<const unsigned long long*>(p->noise_offset_dev);
        fnz.ready = slots + w.noise_counters / sizeof(uint32_t);
        if ((long long)p->B * p->Z >= 0x7fffffffLL || p->Z < 4) { set_error("philox: B*Z=%lld, Z=%d out of range", (long long)p->B * p->Z, p->Z); return 6; }
    }
    ProfScope ps(MPVAE_PROF_PRODUCT_NT, stream);
    // library noise sits on the fp16 grid: one plane, two MMA passes.
    // No tail scratch here: K-slicing the last wave would make the summation order of x = noise.R^T depend on
    // how many rows the call holds, and a row's predictions must not change with the shard it is computed in.
    // nr's rows are padded to 16 bytes inside the workspace: the product may fill the padding with whole-vector stores.
    return tc_gemm_nt(npl, rpl, nr, M, p->L, p->Z, nullptr, slots + SLOT_ABSMAX_R, stream, row_pitch(p->L), p->noise ? 0 : 1,
                      nullptr, 0, jit_noise ? &fnz : nullptr, 1);
}

// CUDA-core regime, up to and including the product: the Philox normals (unless the caller gives the noise) and
// nr = noise . R^T with the FMA engine
int fma_nt_product(const mpvae_probit_params* p, const Workspace& w, cudaStream_t stream) {
    char* base = static_cast<char*>(p->workspace);
    const float* nz = p->noise;
    if (!nz) {
        ProfScope ps(MPVAE_PROF_NOISE, stream);
        float* gen = reinterpret_cast<float*>(base + w.noise_f32);
        if (int rc = launch_philox_normal(gen, p->S, p->B, p->Z, p->noise_b_global, p->noise_row0, p->noise_seed,
                                          p->noise_offset, p->noise_offset_dev, stream)) return rc;
        nz = gen;
    }
    ProfScope ps(MPVAE_PROF_PRODUCT_NT, stream);
    return launch_contract_nt_fma(nz, p->r, reinterpret_cast<float*>(base + w.nr), p->S * p->B, p->L, p->Z, stream,
                                  row_pitch(p->L));
}

// The start of every sampled-prediction entry point: the params in full layout, checked for prediction, and the
// inference layout of mpvae_probit_forward, of which only nr, the noise / R operands and the slots are touched.
// The struct is not copied: p may point at tmp.
struct PredictCall {
    mpvae_probit_params tmp;
    const mpvae_probit_params* p;
    Workspace w;
    RowArgs a;
};

int open_predict(const mpvae_probit_params* p_in, PredictCall& c, bool writes_prob = true) {
    c.p = normalize(p_in, &c.tmp);
    if (!c.p) return 1;
    if (int rc = validate_predict(c.p, writes_prob)) return rc;
    c.w = carve(c.p->S, c.p->B, c.p->L, c.p->Z, false, c.p->flags);
    c.a = row_args(c.p, c.w);
    return 0;
}

// predict's nt product, nr in the workspace: tcgen05 where mpvae_probit_forward takes it for the same
// (S, B, L, Z, flags), the CUDA-core product otherwise
int predict_product(const PredictCall& c, cudaStream_t stream) {
    const mpvae_probit_params* p = c.p;
    if (!use_tensor(p->flags, p->S, p->B, p->L, p->Z)) return fma_nt_product(p, c.w, stream);
    // absmax slot of R, per-block counters of the just-in-time noise
    uint32_t* slots = reinterpret_cast<uint32_t*>(static_cast<char*>(p->workspace) + c.w.slots);
    const cudaError_t e = cudaMemsetAsync(slots, 0, c.w.slots_bytes, stream);
    if (e != cudaSuccess) { set_error("cudaMemsetAsync: %s", cudaGetErrorString(e)); return 2; }
    return dense_nt_product(p, c.w, stream);
}

}  // namespace
}  // namespace mpv

using namespace mpv;

extern "C" {

int mpvae_abi_version(void) { return MPVAE_ABI_VERSION; }
const char* mpvae_last_error(void) { return g_err; }
uint64_t mpvae_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int mpvae_profile(int32_t enable) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.on = enable != 0;
    for (int i = 0; i < MPVAE_PROF_SLOTS; ++i) g_prof.used[i] = 0;
    return 0;
}

int mpvae_profile_read(int32_t slot, double* total_ms, int32_t* count) {
    if (slot < 0 || slot >= MPVAE_PROF_SLOTS || !total_ms || !count) { set_error("profile_read: bad arguments"); return 1; }
    std::lock_guard<std::mutex> lk(g_prof_mu);
    double sum = 0.0;
    for (int i = 0; i < g_prof.used[slot]; ++i) {
        auto& pr = g_prof.pool[slot][i];
        float ms = 0.0f;
        if (cudaEventSynchronize(pr.second) != cudaSuccess || cudaEventElapsedTime(&ms, pr.first, pr.second) != cudaSuccess) {
            set_error("profile_read: event query failed");
            return 2;
        }
        sum += ms;
    }
    *total_ms = sum;
    *count = g_prof.used[slot];
    return 0;
}

const char* mpvae_profile_name(int32_t slot) {
    static const char* names[MPVAE_PROF_SLOTS] = {"noise (philox planes / philox normal / split of an external tensor)",
                                                  "R absmax + split",
                                                  "product nt (noise.R^T)",
                                                  "row forward / finalize",
                                                  "gxs bound",
                                                  "row backward",
                                                  "product tn (g_R)",
                                                  "g_R exchange over peer memory",
                                                  "fused small-regime forward",
                                                  "fused small-regime backward"};
    return (slot >= 0 && slot < MPVAE_PROF_SLOTS) ? names[slot] : nullptr;
}

uint64_t mpvae_workspace_bytes(int32_t S, int32_t B, int32_t L, int32_t Z, int32_t want_backward, uint32_t flags) {
    if (S <= 0 || B <= 0 || L <= 0 || Z <= 0) return 256;
    return carve(S, B, L, Z, want_backward != 0, flags).total;
}

int mpvae_probit_forward(const mpvae_probit_params* p_in, void* cuda_stream) {
    return mpvae_probit_forward_weighted(p_in, nullptr, nullptr, cuda_stream);
}

int mpvae_probit_forward_masked(const mpvae_probit_params* p_in, const uint8_t* label_mask, void* cuda_stream) {
    return mpvae_probit_forward_weighted(p_in, label_mask, nullptr, cuda_stream);
}

int mpvae_probit_forward_weighted(const mpvae_probit_params* p_in, const uint8_t* label_mask, const float* row_weight,
                                  void* cuda_stream) {
    return mpvae_probit_forward_label_weighted(p_in, label_mask, row_weight, nullptr, cuda_stream);
}

// per_row: each p->scalars[k] addresses B floats (one per row) instead of one
static int probit_forward(const mpvae_probit_params* p_in, const uint8_t* label_mask, const float* row_weight,
                          const float* label_weight, bool per_row, void* cuda_stream) {
    mpvae_probit_params tmp;
    const mpvae_probit_params* p = normalize(p_in, &tmp);
    if (!p) return 1;
    if (int rc = validate(p, false)) return rc;
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    // the scratch may be shorter than the backward layout on the inference path; the buffers the forward touches
    // are placed identically in both layouts
    const Workspace w = carve(p->S, p->B, p->L, p->Z, false, p->flags);
    char* base = static_cast<char*>(p->workspace);
    float* nr = reinterpret_cast<float*>(base + w.nr);
    uint32_t* slots = reinterpret_cast<uint32_t*>(base + w.slots);
    cudaError_t e = cudaMemsetAsync(slots, 0, w.slots_bytes, stream);   // last-CTA counter, absmax slots, noise counters
    if (e != cudaSuccess) { set_error("cudaMemsetAsync: %s", cudaGetErrorString(e)); return 2; }
    int rc;
    RowArgs a = row_args(p, w);
    a.mask = label_mask;
    a.row_weight = row_weight;   // read by row_tail only
    a.label_weight = label_weight;
    a.per_row = per_row ? 1 : 0;
    // a scratch block sized for the backward means a training call: the forward keeps E for it (same placement in
    // both layouts: the backward-only buffers follow everything the forward shares)
    const Workspace wb = carve(p->S, p->B, p->L, p->Z, true, p->flags);
    if (p->workspace_bytes >= wb.total) {
        a.E_l = reinterpret_cast<float*>(base + wb.e_l);
        a.E_x = reinterpret_cast<float*>(base + wb.e_x);
    }
    if (use_tensor(p->flags, p->S, p->B, p->L, p->Z)) {
        if ((rc = dense_nt_product(p, w, stream))) return rc;
        ProfScope ps(MPVAE_PROF_ROW_FORWARD, stream);
        return launch_row_forward(a, stream);
    }
    if (use_small(p->flags, p->S, p->B, p->L, p->Z)) {
        // one launch: R staged by TMA, Philox in registers, warp-FMA contraction, row math, per-row tail
        ProfScope ps(MPVAE_PROF_FUSED_SMALL_FWD, stream);
        SmallNoise sn{};
        sn.r = p->r; sn.Z = p->Z;
        sn.noise_ext = p->noise;
        const bool training = a.E_l != nullptr;
        sn.noise_out = (training && !p->noise) ? reinterpret_cast<float*>(base + w.noise_f32) : nullptr;
        sn.nr_out = training ? nr : nullptr;
        sn.Bg = p->noise_b_global; sn.row0 = p->noise_row0;
        sn.seed = p->noise_seed; sn.offset = p->noise_offset; sn.offset_dev = p->noise_offset_dev;
        return launch_small_forward(a, sn, stream);
    }
    if ((rc = fma_nt_product(p, w, stream))) return rc;
    ProfScope ps(MPVAE_PROF_ROW_FORWARD, stream);
    return launch_row_forward(a, stream);
}

int mpvae_probit_forward_label_weighted(const mpvae_probit_params* p_in, const uint8_t* label_mask, const float* row_weight,
                                        const float* label_weight, void* cuda_stream) {
    return probit_forward(p_in, label_mask, row_weight, label_weight, false, cuda_stream);
}

int mpvae_probit_forward_rows(const mpvae_probit_params* p_in, const uint8_t* label_mask, const float* row_weight,
                              const float* label_weight, void* cuda_stream) {
    return probit_forward(p_in, label_mask, row_weight, label_weight, true, cuda_stream);
}

int mpvae_probit_predict(const mpvae_probit_params* p_in, void* cuda_stream) {
    PredictCall c;
    if (int rc = open_predict(p_in, c)) return rc;
    const mpvae_probit_params* p = c.p;
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    if (use_small(p->flags, p->S, p->B, p->L, p->Z)) {
        ProfScope ps(MPVAE_PROF_FUSED_SMALL_FWD, stream);
        SmallNoise sn{};
        sn.r = p->r; sn.Z = p->Z;
        sn.noise_ext = p->noise;
        sn.Bg = p->noise_b_global; sn.row0 = p->noise_row0;
        sn.seed = p->noise_seed; sn.offset = p->noise_offset; sn.offset_dev = p->noise_offset_dev;
        return launch_small_predict(c.a, sn, stream);
    }
    if (int rc = predict_product(c, stream)) return rc;
    ProfScope ps(MPVAE_PROF_ROW_FORWARD, stream);
    return launch_predict_rows(c.a, stream);
}

int mpvae_probit_predict_conditional(const mpvae_probit_params* p_in, const int8_t* observed, float* log_evidence,
                                     float* ess, void* cuda_stream) {
    PredictCall c;
    if (int rc = open_predict(p_in, c)) return rc;
    if (!observed || !log_evidence || !ess) { set_error("NULL pointer (observed/log_evidence/ess)"); return 1; }
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    FusePart* part = reinterpret_cast<FusePart*>(static_cast<char*>(c.p->workspace) + c.w.fuse_part);
    // the CUDA-core product also where predict takes the one-launch small kernel, which never materialises nr (its
    // forward outputs equal the CUDA-core path's bit for bit)
    if (int rc = predict_product(c, stream)) return rc;
    ProfScope ps(MPVAE_PROF_ROW_FORWARD, stream);
    return launch_conditional_rows(c.a, observed, part, log_evidence, ess, stream);
}

int mpvae_probit_sample_labels(const mpvae_probit_params* p_in, const float* uniform, int32_t* bits, void* cuda_stream) {
    PredictCall c;
    if (int rc = open_predict(p_in, c, false)) return rc;
    const mpvae_probit_params* p = c.p;
    if (!bits) { set_error("NULL pointer (bits)"); return 1; }
    if (int rc = check_rows_fit(p, !uniform, "label draws")) return rc;
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    // the CUDA-core product also where predict takes the one-launch small kernel, which never materialises nr
    if (int rc = predict_product(c, stream)) return rc;
    const SampleInputs in{uniform, bits, philox_rows(p)};
    ProfScope ps(MPVAE_PROF_ROW_FORWARD, stream);
    return launch_sample_labels(c.a, in, stream);
}

uint64_t mpvae_f1_sets_workspace_bytes(int32_t B, int32_t S, int32_t L) {
    if (B <= 0 || S <= 0 || L <= 0) return 256;
    return f1_layout(B, S, L).total;
}

int mpvae_f1_sets(const int32_t* bits, int32_t B, int32_t S, int32_t L, double beta, int32_t max_size, uint8_t* sets,
                  double* expected_f, int32_t* set_size, void* ws, uint64_t ws_bytes, void* cuda_stream) {
    if (B <= 0 || S <= 0 || L <= 0) {
        set_error("bad sizes B=%d S=%d L=%d (empty batches are handled by the host wrapper)", B, S, L);
        return 1;
    }
    if (!(beta > 0.0) || !isfinite(beta * beta)) {   // beta^2 enters every weight: it must be finite too
        set_error("beta=%g must be positive with a finite square", beta);
        return 1;
    }
    if (max_size < 0) { set_error("max_size=%d must be >= 0", max_size); return 1; }
    if (!bits || !sets || !expected_f || !set_size || !ws) {
        set_error("NULL pointer (bits/sets/expected_f/set_size/ws)");
        return 1;
    }
    if (int rc = check_scratch("f1 sets workspace", ws, ws_bytes, mpvae_f1_sets_workspace_bytes(B, S, L))) return rc;
    return launch_f1_sets(bits, B, S, L, beta, max_size, sets, expected_f, set_size, ws, static_cast<cudaStream_t>(cuda_stream));
}

uint64_t mpvae_mode_workspace_bytes(int32_t S, int32_t B, int32_t L) {
    if (S <= 0 || B <= 0 || L <= 0) return 256;
    return mode_layout(S, B, L).total;
}

int mpvae_probit_score_sets(const mpvae_probit_params* p_in, const int32_t* bits, int32_t C, double* log_prob,
                            double* ess, void* mode_ws, uint64_t mode_ws_bytes, void* cuda_stream) {
    PredictCall c;
    if (int rc = open_predict(p_in, c, false)) return rc;
    if (!bits || !log_prob || !ess) { set_error("NULL pointer (bits/log_prob/ess)"); return 1; }
    if (C <= 0) { set_error("bad set count C=%d", C); return 1; }
    if ((long long)c.p->B * C > 0x7fffffffLL) { set_error("B*C overflows int32"); return 1; }
    if (int rc = check_scratch("mode_ws", mode_ws, mode_ws_bytes, mpvae_mode_workspace_bytes(c.p->S, c.p->B, c.p->L))) return rc;
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    // the CUDA-core product also where predict takes the one-launch small kernel, which never materialises nr
    if (int rc = predict_product(c, stream)) return rc;
    ProfScope ps(MPVAE_PROF_ROW_FORWARD, stream);
    return launch_score_sets(c.a, bits, C, log_prob, ess, mode_ws, stream);
}

int mpvae_probit_predict_mode(const mpvae_probit_params* p_in, int32_t max_flips, uint8_t* sets, double* log_prob,
                              double* ess, int32_t* size, int32_t* flips, void* mode_ws, uint64_t mode_ws_bytes,
                              void* cuda_stream) {
    PredictCall c;
    if (int rc = open_predict(p_in, c, false)) return rc;
    if (!sets || !log_prob || !ess || !size || !flips) { set_error("NULL pointer (sets/log_prob/ess/size/flips)"); return 1; }
    if (max_flips < 0) { set_error("max_flips=%d must be >= 0", max_flips); return 1; }
    if (int rc = check_scratch("mode_ws", mode_ws, mode_ws_bytes, mpvae_mode_workspace_bytes(c.p->S, c.p->B, c.p->L))) return rc;
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    if (int rc = predict_product(c, stream)) return rc;
    ProfScope ps(MPVAE_PROF_ROW_FORWARD, stream);
    return launch_predict_mode(c.a, max_flips, sets, log_prob, ess, size, flips, mode_ws, stream);
}

// G = R R^T takes the engine its own (L, L, Z) shape selects, as mpvae_contract_nt's auto engine does, unless
// MPVAE_FLAG_CONTRACT_FMA asks for the CUDA-core product
static bool gram_uses_tensor(uint32_t flags, int L, int Z) {
    return !(flags & MPVAE_FLAG_CONTRACT_FMA) && use_tensor(0, 1, L, L, Z);
}

static GhkLayout ghk_layout_for(int S, int B, int L, int Z, int mo, uint32_t flags) {
    return ghk_layout(S, B, L, mo, gram_uses_tensor(flags, L, Z) ? tc_workspace_nt(L, L, Z) : 0);
}

uint64_t mpvae_ghk_workspace_bytes(int32_t S, int32_t B, int32_t L, int32_t Z, int32_t max_observed, uint32_t flags) {
    if (S <= 0 || B <= 0 || L <= 0 || Z <= 0 || max_observed < 0 || max_observed > L) return 256;
    return ghk_layout_for(S, B, L, Z, max_observed, flags).total;
}

int mpvae_probit_predict_conditional_ghk(const mpvae_probit_params* p_in, const int8_t* observed, const float* gram,
                                         const float* zeta, const float* uniform, void* ghk_ws, uint64_t ghk_ws_bytes,
                                         int32_t max_observed, float* log_evidence, float* ess, void* cuda_stream) {
    PredictCall c;
    if (int rc = open_predict(p_in, c)) return rc;
    const mpvae_probit_params* p = c.p;
    if (!observed || !log_evidence || !ess || !ghk_ws) { set_error("NULL pointer (observed/log_evidence/ess/ghk_ws)"); return 1; }
    if (max_observed < 0 || max_observed > p->L) { set_error("max_observed=%d outside [0, L=%d]", max_observed, p->L); return 1; }
    const GhkLayout gl = ghk_layout_for(p->S, p->B, p->L, p->Z, max_observed, p->flags);
    char sized_for[32];
    snprintf(sized_for, sizeof(sized_for), "max_observed=%d", max_observed);
    if (int rc = check_scratch("ghk workspace", ghk_ws, ghk_ws_bytes, gl.total, sized_for)) return rc;
    if (int rc = check_rows_fit(p, !zeta || !uniform, "GHK draws")) return rc;
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    char* gbase = static_cast<char*>(ghk_ws);
    int rc;
    if (!gram && max_observed > 0) {
        float* G = reinterpret_cast<float*>(gbase + gl.gram);
        rc = gram_uses_tensor(p->flags, p->L, p->Z)
                 ? tc_contract_nt(p->r, p->r, G, p->L, p->L, p->Z, gbase + gl.gram_scratch, tc_workspace_nt(p->L, p->L, p->Z), stream)
                 : launch_contract_nt_fma(p->r, p->r, G, p->L, p->L, p->Z, stream);
        if (rc) return rc;
        gram = G;
    }
    if ((rc = predict_product(c, stream))) return rc;
    const GhkInputs in{gl, ghk_ws, max_observed, observed, gram, zeta, uniform, philox_rows(p), log_evidence, ess};
    ProfScope ps(MPVAE_PROF_ROW_FORWARD, stream);
    return launch_ghk_rows(c.a, in, stream);
}

int mpvae_probit_backward(const mpvae_probit_params* p_in, void* cuda_stream) {
    return mpvae_probit_backward_weighted(p_in, nullptr, nullptr, cuda_stream);
}

int mpvae_probit_backward_masked(const mpvae_probit_params* p_in, const uint8_t* label_mask, void* cuda_stream) {
    return mpvae_probit_backward_weighted(p_in, label_mask, nullptr, cuda_stream);
}

int mpvae_probit_backward_weighted(const mpvae_probit_params* p_in, const uint8_t* label_mask, const float* row_weight,
                                   void* cuda_stream) {
    return mpvae_probit_backward_label_weighted(p_in, label_mask, row_weight, nullptr, cuda_stream);
}

// per_row: each p->g_scalars[k] addresses B floats (one cotangent per row) or is NULL
static int probit_backward(const mpvae_probit_params* p_in, const uint8_t* label_mask, const float* row_weight,
                           const float* label_weight, bool per_row, void* cuda_stream) {
    mpvae_probit_params tmp;
    const mpvae_probit_params* p = normalize(p_in, &tmp);
    if (!p) return 1;
    if (int rc = validate(p, true)) return rc;
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    const Workspace w = carve(p->S, p->B, p->L, p->Z, true, p->flags);
    char* base = static_cast<char*>(p->workspace);
    uint32_t* slots = reinterpret_cast<uint32_t*>(base + w.slots);
    const bool tensor = use_tensor(p->flags, p->S, p->B, p->L, p->Z);
    RowArgs a = row_args(p, w);
    a.mask = label_mask;
    a.row_weight = row_weight;   // scales the per-row coefficients, and with them the gxs bound of the fp16 planes
    a.label_weight = label_weight;
    a.per_row = per_row ? 1 : 0;   // row b's cotangents: they enter the gxs bound through row_coeffs as well
    a.E_l = reinterpret_cast<float*>(base + w.e_l);
    a.E_x = reinterpret_cast<float*>(base + w.e_x);
    const int M = p->S * p->B;
    if (p->g_r && tensor) {
        // slots 2..5: scale source of the gxs planes, max |g_indiv_prob|, max |g_indiv_prob_label|, max |label weight|
        if (cudaMemsetAsync(slots + SLOT_ABSMAX_GXS, 0, 4 * sizeof(uint32_t), stream) != cudaSuccess) { set_error("cudaMemsetAsync failed"); return 2; }
        // the plane scale comes from an upper bound of |gxs| computed from the saved row statistics, so the row
        // kernel can write the operand planes itself
        ProfScope ps(MPVAE_PROF_GXS_BOUND, stream);
        if (p->g_indiv_prob) { if (int rc = tc_absmax(p->g_indiv_prob, (size_t)p->B * p->L, slots + SLOT_ABSMAX_GP, stream)) return rc; }
        if (p->g_indiv_prob_label) { if (int rc = tc_absmax(p->g_indiv_prob_label, (size_t)p->B * p->L, slots + SLOT_ABSMAX_GP + 1, stream)) return rc; }
        if (label_weight) { if (int rc = tc_absmax(label_weight, (size_t)2 * p->L, slots + SLOT_ABSMAX_LW, stream)) return rc; }
        if (int rc = launch_gxs_bound(a, slots + SLOT_ABSMAX_GP, slots + SLOT_ABSMAX_GXS, slots + SLOT_ABSMAX_LW, stream)) return rc;
        a.gxs_planes = reinterpret_cast<__half*>(base + w.gxs_planes);
        a.gxs_pitch = tc_pitch(p->L);
        a.gxs_plane_elems = (size_t)M * a.gxs_pitch;
        a.gxs_scale = slots + SLOT_ABSMAX_GXS;
    } else if (p->g_r) {
        a.gxs = reinterpret_cast<float*>(base + w.gxs);
    }
    const bool small = use_small(p->flags, p->S, p->B, p->L, p->Z);
    if (!small) {
        ProfScope ps(MPVAE_PROF_ROW_BACKWARD, stream);
        if (int rc = launch_row_backward(a, stream)) return rc;
    }
    if (!p->g_r && !small) return 0;
    // data-parallel: the product writes this rank's partial into its own `part` buffer, peer_reduce.cu sums the world's
    // partials over NVLink and leaves the result in every rank's g_r
    const bool peer = p->peer_world > 1 && p->g_r != nullptr;
    PeerCtx pctx{};
    float* g_r_out = p->g_r;
    if (peer) {
        if (p->peer_world > 8 || p->peer_rank < 0 || p->peer_rank >= p->peer_world || p->peer_step == 0 ||
            p->g_r != p->peer_g_r[p->peer_rank]) {
            set_error("peer tables: world %d rank %d step %u (g_r must be peer_g_r[rank])", p->peer_world, p->peer_rank, p->peer_step);
            return 1;
        }
        pctx.world = p->peer_world; pctx.rank = p->peer_rank; pctx.step = p->peer_step;
        pctx.step_dev = p->peer_step_dev; pctx.step_stride = 1;
        pctx.timeout_cycles = peer_timeout_cycles();
        for (int i = 0; i < p->peer_world; ++i) {
            pctx.part[i] = static_cast<float*>(p->peer_part[i]);
            pctx.g_r[i] = static_cast<float*>(p->peer_g_r[i]);
            pctx.flags[i] = static_cast<uint32_t*>(p->peer_flags[i]);
            if (!pctx.part[i] || !pctx.g_r[i] || !pctx.flags[i]) { set_error("peer tables: NULL entry for rank %d", i); return 1; }
        }
        g_r_out = pctx.part[p->peer_rank];
    }
    if (small) {
        // one CTA per row (cells from the kept E / nr, logit and KL gradients, the row's share of g_R), then the
        // deterministic sum of the shares over the batch
        ProfScope ps(MPVAE_PROF_FUSED_SMALL_BWD, stream);
        SmallNoise sn{};
        sn.r = p->r; sn.Z = p->Z;
        sn.noise_ext = p->noise;
        sn.noise_out = reinterpret_cast<float*>(base + w.noise_f32);
        sn.partial = p->g_r ? reinterpret_cast<float*>(base + w.small_partials) : nullptr;
        if (int rc = launch_small_backward(a, sn, p->g_r ? g_r_out : nullptr, stream)) return rc;
        if (!p->g_r) return 0;
    } else {
        ProfScope ps(MPVAE_PROF_PRODUCT_TN, stream);
        int rc;
        if (tensor) {
            // data-parallel: the product publishes its finished tiles in per-tile counters (tc_warps.cuh), and the exchange
            // sums them over the ranks slab by slab on a few reserved SMs beside the product -- unless the product is too
            // short to hide it (measured) or the caller asks for the exchange after the product
            FusePeer fp{};
            const bool tiles_ok = peer && p->peer_tile_done[p->peer_rank] != nullptr && !(p->peer_mc_part && p->peer_mc_g_r) &&
                                  (size_t)ceil_div(p->L, 256) * ceil_div(p->Z, 256) < kTileEpochWord;
            const bool beside = tiles_ok && !(p->flags & MPVAE_FLAG_SERIAL_EXCHANGE) && ceil_div(p->Z, 256) <= 32 &&
                                p->L >= 512 && (long long)p->S * p->B >= 8192;
            SideStream* side = nullptr;
            PeerCtx sctx = pctx;                                 // the slab exchange: flag value = the tile epoch
            if (beside) {
                for (int i = 0; i < pctx.world; ++i)
                    if (!p->peer_tile_done[i]) { set_error("peer tables: NULL tile counters for rank %d", i); return 1; }
                side = side_stream();
                if (!side) return 2;
                if (cudaEventRecord(side->fork, stream) != cudaSuccess || cudaStreamWaitEvent(side->stream, side->fork, 0) != cudaSuccess) {
                    set_error("peer: fork failed");
                    return 2;
                }
                uint32_t* epoch_word = static_cast<uint32_t*>(p->peer_tile_done[p->peer_rank]) + kTileEpochWord;
                sctx.step = 1; sctx.step_dev = epoch_word; sctx.step_stride = 0;
                pctx.epoch_dev = epoch_word;                     // advanced by the closing flag phase below
                fp.world = pctx.world;
                fp.done = static_cast<unsigned int*>(p->peer_tile_done[p->peer_rank]);
            }
            int exchanged = 0;
            // the noise planes the forward left in the workspace are the MN-major B operand as they are
            rc = tc_gemm_tn(base + w.gxs_planes, base + w.noise_planes, g_r_out, M, p->L, p->Z, slots + SLOT_ABSMAX_GXS, nullptr, stream,
                            p->noise ? 0 : 1, base + w.tn_tail, tc_tail_scratch_bytes(), 0, beside ? &fp : nullptr, &exchanged);
            if (rc) return rc;
            if (beside) {
                // the complete 256-row slabs among the exchanged tiles go over NVLink beside the product, on the SMs it left free
                // (only slabs of a full 256 rows: a partial last slab goes with the tail rows)
                const int tiles_n = ceil_div(p->Z, 256);
                int n_slabs = exchanged / tiles_n;
                if (n_slabs > p->L / 256) n_slabs = p->L / 256;
                if (int rc2 = launch_peer_reduce_slabs(sctx, p->peer_tile_done, tiles_n, n_slabs, (size_t)256 * p->Z,
                                                       exchange_sms(p->peer_world), side->stream)) return rc2;
                if (cudaEventRecord(side->join, side->stream) != cudaSuccess || cudaStreamWaitEvent(stream, side->join, 0) != cudaSuccess) {
                    set_error("peer: join failed");
                    return 2;
                }
                // what is left: the rows of the K-sliced tail tiles (complete only now, after the fix-up kernel), and the
                // two flag phases that tell every rank that all deliveries of this step have landed
                const size_t first_row = (size_t)n_slabs * 256;
                const size_t first = first_row < (size_t)p->L ? first_row * p->Z : (size_t)p->L * p->Z;
                ProfScope px(MPVAE_PROF_EXCHANGE, stream);
                return launch_peer_reduce(pctx, (size_t)p->L * p->Z - first, stream, first);
            }
        } else {
            const float* nz = p->noise ? p->noise : reinterpret_cast<const float*>(base + w.noise_f32);
            rc = launch_contract_tn_fma(a.gxs, nz, g_r_out, M, p->L, p->Z, base + w.fma_partials, w.total - w.fma_partials, stream,
                                        row_pitch(p->L));
        }
        if (rc) return rc;
    }
    if (!peer) return 0;
    ProfScope ps(MPVAE_PROF_EXCHANGE, stream);
    if (p->peer_mc_part && p->peer_mc_g_r)
        return launch_peer_reduce_nvls(pctx, static_cast<const float*>(p->peer_mc_part), static_cast<float*>(p->peer_mc_g_r),
                                       (size_t)p->L * p->Z, stream);
    return launch_peer_reduce(pctx, (size_t)p->L * p->Z, stream);
}

int mpvae_probit_backward_label_weighted(const mpvae_probit_params* p_in, const uint8_t* label_mask, const float* row_weight,
                                         const float* label_weight, void* cuda_stream) {
    return probit_backward(p_in, label_mask, row_weight, label_weight, false, cuda_stream);
}

int mpvae_probit_backward_rows(const mpvae_probit_params* p_in, const uint8_t* label_mask, const float* row_weight,
                               const float* label_weight, void* cuda_stream) {
    return probit_backward(p_in, label_mask, row_weight, label_weight, true, cuda_stream);
}

int mpvae_test_log_normal(const float* in, float* out, float* ref, uint64_t n, void* cuda_stream) {
    if (!in || !out || !ref || n == 0) { set_error("test_log_normal: bad arguments"); return 1; }
    return launch_log_normal_probe(in, out, ref, (size_t)n, static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_test_erf(const float* in, float* out, float* ref, uint64_t n, void* cuda_stream) {
    if (!in || !out || !ref || n == 0) { set_error("test_erf: bad arguments"); return 1; }
    return launch_erf_probe(in, out, ref, (size_t)n, static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_test_warp_sum(const void* in, void* out, void* ref, int32_t groups, int32_t fp64, void* cuda_stream) {
    if (!in || !out || !ref || groups <= 0) { set_error("test_warp_sum: bad arguments"); return 1; }
    return launch_warp_sum_probe(in, out, ref, groups, fp64 != 0, static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_philox_normal(float* noise, int32_t S, int32_t B, int32_t Z, int32_t B_global, int32_t row0, uint64_t seed,
                        uint64_t offset, void* cuda_stream) {
    if (!noise) { set_error("philox: NULL output"); return 1; }
    if (S < 0 || B < 0 || Z < 0 || row0 < 0 || B_global < row0 + B) {
        set_error("philox: bad sizes S=%d B=%d Z=%d B_global=%d row0=%d", S, B, Z, B_global, row0);
        return 1;
    }
    return launch_philox_normal(noise, S, B, Z, B_global, row0, seed, offset, nullptr, static_cast<cudaStream_t>(cuda_stream));
}

uint64_t mpvae_batch_metrics_workspace(int32_t B, int32_t L) {
    if (B <= 0 || L <= 0) return 256;
    return batch_metrics_workspace(B, L);
}

int mpvae_batch_metrics(const float* indiv_prob, const float* input_label, int32_t B, int32_t L, float threshold, double* out,
                        void* workspace, uint64_t workspace_bytes, void* cuda_stream) {
    if (!indiv_prob || !input_label || !out || !workspace || B <= 0 || L <= 0) { set_error("batch_metrics: bad arguments"); return 1; }
    if (workspace_bytes < batch_metrics_workspace(B, L)) { set_error("batch_metrics: workspace too small"); return 1; }
    return launch_batch_metrics(indiv_prob, input_label, B, L, threshold, out, workspace, static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_predictive_scale(const float* r, int32_t L, int32_t Z, double* scale_out, void* cuda_stream) {
    if (!r || !scale_out) { set_error("predictive_scale: NULL pointer (r/scale_out)"); return 1; }
    if (L <= 0 || Z <= 0) { set_error("predictive_scale: bad sizes L=%d Z=%d", L, Z); return 1; }
    return launch_predictive_scale(r, L, Z, scale_out, static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_predictive_rho(const float* r, int32_t L, int32_t Z, const double* scale, const int32_t* pairs, int32_t P,
                         double* rho_out, void* cuda_stream) {
    if (!r || !scale || !pairs || !rho_out) { set_error("predictive_rho: NULL pointer (r/scale/pairs/rho_out)"); return 1; }
    if (L <= 0 || Z <= 0 || P < 0) { set_error("predictive_rho: bad sizes L=%d Z=%d P=%d", L, Z, P); return 1; }
    if (reinterpret_cast<uintptr_t>(pairs) & 7u) { set_error("predictive_rho: pairs must be 8-byte aligned"); return 1; }
    return launch_predictive_rho(r, L, Z, scale, pairs, P, rho_out, static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_predict_exact(const float* fx_out, int32_t B, int32_t L, const double* scale, uint32_t flags, float* indiv_prob,
                        void* cuda_stream) {
    if (!fx_out || !scale || !indiv_prob) { set_error("predict_exact: NULL pointer (fx_out/scale/indiv_prob)"); return 1; }
    if (B < 0 || L <= 0) { set_error("predict_exact: bad sizes B=%d L=%d", B, L); return 1; }
    return launch_predict_exact(fx_out, B, L, scale, (flags & MPVAE_FLAG_STABLE_CDF) != 0, indiv_prob,
                                static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_predict_pairs(const float* fx_out, int32_t B, int32_t L, const double* scale, const int32_t* pairs,
                        const double* rho, int32_t P, uint32_t flags, float* out, void* cuda_stream) {
    if (!fx_out || !scale || !pairs || !rho || !out) { set_error("predict_pairs: NULL pointer (fx_out/scale/pairs/rho/out)"); return 1; }
    if (B < 0 || L <= 0 || P < 0) { set_error("predict_pairs: bad sizes B=%d L=%d P=%d", B, L, P); return 1; }
    if (reinterpret_cast<uintptr_t>(pairs) & 7u) { set_error("predict_pairs: pairs must be 8-byte aligned"); return 1; }
    return launch_predict_pairs(fx_out, B, L, scale, pairs, rho, P, (flags & MPVAE_FLAG_STABLE_CDF) != 0, out,
                                static_cast<cudaStream_t>(cuda_stream));
}

uint64_t mpvae_contract_workspace_bytes(int32_t M, int32_t N, int32_t K, int32_t engine) {
    // covers both orientations: nt (M,N,K) and tn (M = reduction, N1 = N, N2 = K)
    size_t a = contract_tn_fma_workspace(M, N, K);
    engine &= ~MPVAE_ENGINE_KSPLIT;
    if (engine != 1 && tc_available()) {
        size_t t1 = tc_workspace_nt(M, N, K), t2 = tc_workspace_tn(M, N, K);
        if (t1 > a) a = t1;
        if (t2 > a) a = t2;
    }
    return align_up(a, 256) + 256;
}

int mpvae_contract_nt(const float* A, const float* Bm, float* C, int32_t M, int32_t N, int32_t K, int32_t engine,
                      void* workspace, uint64_t workspace_bytes, void* cuda_stream) {
    return mpvae_contract_nt_pitched(A, Bm, C, M, N, K, N, engine, workspace, workspace_bytes, cuda_stream);
}

int mpvae_contract_nt_pitched(const float* A, const float* Bm, float* C, int32_t M, int32_t N, int32_t K, int32_t ldc,
                              int32_t engine, void* workspace, uint64_t workspace_bytes, void* cuda_stream) {
    if (!A || !Bm || !C || M <= 0 || N <= 0 || K <= 0 || ldc < N) { set_error("contract_nt: bad arguments"); return 1; }
    const int ksplit = (engine & MPVAE_ENGINE_KSPLIT) ? 1 : 0;
    engine &= ~MPVAE_ENGINE_KSPLIT;
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    if (engine == 0) engine = use_tensor(0, 1, M, N, K) ? 2 : 1;
    if (engine >= 2 && engine <= 5) {
        if (!tc_available()) { set_error("contract_nt: tensor engine not built"); return 7; }
        return tc_contract_nt(A, Bm, C, M, N, K, workspace, workspace_bytes, stream, engine == 3 || engine == 5, engine >= 4, ldc,
                              ksplit);
    }
    return launch_contract_nt_fma(A, Bm, C, M, N, K, stream, ldc);
}

int mpvae_contract_tn(const float* A, const float* Bm, float* C, int32_t M, int32_t N1, int32_t N2, int32_t engine,
                      void* workspace, uint64_t workspace_bytes, void* cuda_stream) {
    if (!A || !Bm || !C || M <= 0 || N1 <= 0 || N2 <= 0) { set_error("contract_tn: bad arguments"); return 1; }
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    if (engine == 0) engine = use_tensor(0, 1, M, N1, N2) ? 2 : 1;
    if (engine >= 2 && engine <= 5) {
        if (!tc_available()) { set_error("contract_tn: tensor engine not built"); return 7; }
        return tc_contract_tn(A, Bm, C, M, N1, N2, workspace, workspace_bytes, stream, engine == 3 || engine == 5, engine >= 4);
    }
    return launch_contract_tn_fma(A, Bm, C, M, N1, N2, workspace, workspace_bytes, stream);
}

// ---- peer memory (CUDA IPC).  The 64-byte handle is cudaIpcMemHandle_t; allocations are made with cudaMalloc so that
// the handle addresses exactly the buffer (no sub-allocation offsets). ----
uint64_t mpvae_peer_flag_bytes(void) { return peer_flag_bytes(); }

int mpvae_peer_allreduce_dev(void* const* part, void* const* g_r, void* const* flags, int32_t world, int32_t rank, uint32_t step,
                             uint32_t* step_dev, uint64_t n, void* cuda_stream) {
    if (!part || !g_r || !flags || world < 2 || world > 8 || rank < 0 || rank >= world || step == 0 || n == 0) {
        set_error("peer_allreduce: bad arguments");
        return 1;
    }
    PeerCtx ctx{};
    ctx.world = world; ctx.rank = rank; ctx.step = step;
    ctx.step_dev = step_dev; ctx.step_stride = 1;
    ctx.timeout_cycles = peer_timeout_cycles();
    for (int i = 0; i < world; ++i) {
        ctx.part[i] = static_cast<float*>(part[i]);
        ctx.g_r[i] = static_cast<float*>(g_r[i]);
        ctx.flags[i] = static_cast<uint32_t*>(flags[i]);
        if (!ctx.part[i] || !ctx.g_r[i] || !ctx.flags[i]) { set_error("peer_allreduce: NULL table entry %d", i); return 1; }
        if ((reinterpret_cast<uintptr_t>(ctx.part[i]) | reinterpret_cast<uintptr_t>(ctx.g_r[i])) & 15) {
            set_error("peer_allreduce: table entry %d is not 16-byte aligned", i);
            return 1;
        }
    }
    return launch_peer_reduce(ctx, (size_t)n, static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_peer_allreduce(void* const* part, void* const* g_r, void* const* flags, int32_t world, int32_t rank, uint32_t step,
                         uint64_t n, void* cuda_stream) {
    return mpvae_peer_allreduce_dev(part, g_r, flags, world, rank, step, nullptr, n, cuda_stream);
}

int mpvae_peer_allreduce_nvls(void* const* part, void* const* g_r, void* const* flags, void* mc_part, void* mc_g_r, int32_t world,
                              int32_t rank, uint32_t step, uint64_t n, void* cuda_stream) {
    if (!part || !g_r || !flags || !mc_part || !mc_g_r || world < 2 || world > 8 || rank < 0 || rank >= world || step == 0 || n == 0) {
        set_error("peer_allreduce_nvls: bad arguments");
        return 1;
    }
    PeerCtx ctx{};
    ctx.world = world; ctx.rank = rank; ctx.step = step;
    ctx.timeout_cycles = peer_timeout_cycles();
    for (int i = 0; i < world; ++i) {
        ctx.part[i] = static_cast<float*>(part[i]);
        ctx.g_r[i] = static_cast<float*>(g_r[i]);
        ctx.flags[i] = static_cast<uint32_t*>(flags[i]);
        if (!ctx.part[i] || !ctx.g_r[i] || !ctx.flags[i]) { set_error("peer_allreduce_nvls: NULL table entry %d", i); return 1; }
    }
    return launch_peer_reduce_nvls(ctx, static_cast<const float*>(mc_part), static_cast<float*>(mc_g_r), (size_t)n,
                                   static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_peer_error(const void* flags, uint32_t* out_step, void* cuda_stream) {
    if (!flags || !out_step) { set_error("peer_error: bad arguments"); return 1; }
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    const cudaError_t e = cudaMemcpyAsync(out_step, static_cast<const uint32_t*>(flags) + peer_error_word(), sizeof(uint32_t),
                                          cudaMemcpyDeviceToHost, stream);
    if (e != cudaSuccess || cudaStreamSynchronize(stream) != cudaSuccess) { set_error("peer_error: copy failed"); return 2; }
    return 0;
}

int mpvae_peer_alloc(uint64_t bytes, void** ptr, unsigned char handle[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    if (!ptr || !handle || bytes == 0) { set_error("peer_alloc: bad arguments"); return 1; }
    cudaError_t e = cudaMalloc(ptr, bytes);
    if (e != cudaSuccess) { set_error("peer_alloc: cudaMalloc(%llu): %s", (unsigned long long)bytes, cudaGetErrorString(e)); return 2; }
    e = cudaMemset(*ptr, 0, bytes);
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle), *ptr);
    if (e != cudaSuccess) { set_error("peer_alloc: %s", cudaGetErrorString(e)); cudaFree(*ptr); *ptr = nullptr; return 2; }
    return 0;
}

int mpvae_peer_open(const unsigned char handle[64], void** ptr) {
    if (!ptr || !handle) { set_error("peer_open: bad arguments"); return 1; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    const cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { set_error("peer_open: cudaIpcOpenMemHandle: %s", cudaGetErrorString(e)); return 2; }
    return 0;
}

int mpvae_peer_close(void* ptr) {
    if (ptr && cudaIpcCloseMemHandle(ptr) != cudaSuccess) { set_error("peer_close failed"); return 2; }
    return 0;
}

int mpvae_peer_free(void* ptr) {
    if (ptr && cudaFree(ptr) != cudaSuccess) { set_error("peer_free failed"); return 2; }
    return 0;
}

uint64_t mpvae_tc_planes_bytes(int32_t rows, int32_t cols) { return (rows > 0 && cols > 0) ? tc_planes_bytes(rows, cols) : 0; }
uint64_t mpvae_tc_tail_scratch_bytes(void) { return tc_tail_scratch_bytes(); }

int mpvae_tc_split(const float* src, int32_t rows, int32_t cols, void* planes, uint32_t* absmax_slot, void* cuda_stream) {
    if (!src || !planes || !absmax_slot || rows <= 0 || cols < 8) { set_error("tc_split: bad arguments"); return 1; }
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    if (cudaMemsetAsync(absmax_slot, 0, sizeof(uint32_t), stream) != cudaSuccess) { set_error("cudaMemsetAsync failed"); return 2; }
    return tc_split(src, rows, cols, planes, absmax_slot, 1, stream);
}

int mpvae_tc_gemm_nt(const void* a_planes, const void* b_planes, float* C, int32_t M, int32_t N, int32_t K, int32_t ldc,
                     const uint32_t* absmax_a, const uint32_t* absmax_b, int32_t ksplit, void* tail_scratch,
                     uint64_t tail_scratch_bytes, void* cuda_stream) {
    if (!a_planes || !b_planes || !C || M <= 0 || N <= 0 || K <= 0 || (ldc != 0 && ldc < N)) { set_error("tc_gemm_nt: bad arguments"); return 1; }
    return tc_gemm_nt(a_planes, b_planes, C, M, N, K, absmax_a, absmax_b, static_cast<cudaStream_t>(cuda_stream), ldc, 0,
                      ksplit ? tail_scratch : nullptr, ksplit ? (size_t)tail_scratch_bytes : 0);
}

int mpvae_tc_gemm_tn(const void* a_planes, const void* b_planes, float* C, int32_t M, int32_t N1, int32_t N2,
                     const uint32_t* absmax_a, const uint32_t* absmax_b, void* tail_scratch, uint64_t tail_scratch_bytes,
                     void* cuda_stream) {
    if (!a_planes || !b_planes || !C || M <= 0 || N1 <= 0 || N2 <= 0) { set_error("tc_gemm_tn: bad arguments"); return 1; }
    return tc_gemm_tn(a_planes, b_planes, C, M, N1, N2, absmax_a, absmax_b, static_cast<cudaStream_t>(cuda_stream), 0,
                      tail_scratch, (size_t)tail_scratch_bytes);
}

int mpvae_label_curves(const float* sorted_scores, const float* sorted_targets, int32_t N, int32_t L, double fdr_cutoff,
                       double* out, void* cuda_stream) {
    if (!sorted_scores || !sorted_targets || !out || N <= 0 || L <= 0) { set_error("label_curves: bad arguments"); return 1; }
    return launch_label_curves(sorted_scores, sorted_targets, N, L, fdr_cutoff, out, static_cast<cudaStream_t>(cuda_stream));
}

uint64_t mpvae_grad_norm_workspace(void) { return grad_norm_workspace(); }

int mpvae_grad_norm(const float* g, uint64_t n, double max_norm, double grad_scale, const float* lr_dev, double lr, double beta1,
                    double beta2, double* state, void* workspace, uint64_t workspace_bytes, void* cuda_stream) {
    if (!g || !state || !workspace || workspace_bytes < grad_norm_workspace()) { set_error("grad_norm: bad arguments"); return 1; }
    return launch_grad_norm(g, (size_t)n, workspace, max_norm, grad_scale, lr_dev, lr, beta1, beta2, state,
                            static_cast<cudaStream_t>(cuda_stream));
}

int mpvae_adam_step(void* p, int32_t p_is_f64, const float* g, void* m, void* v, float* shadow_f32, uint64_t n,
                    const double* state, double beta1, double beta2, double eps, double weight_decay, void* cuda_stream) {
    if (!p || !g || !m || !v || !state) { set_error("adam_step: NULL pointer"); return 1; }
    return launch_adam(p, p_is_f64, g, m, v, shadow_f32, (size_t)n, state, beta1, beta2, eps, weight_decay,
                       static_cast<cudaStream_t>(cuda_stream));
}

}  // extern "C"
