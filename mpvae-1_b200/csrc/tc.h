// tcgen05 (5th-gen tensor core) contraction engine: split-precision GEMMs for the dense regime (label / rank sets
// >= 128).  See contract_tc.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace mpv {

struct FuseNoise;   // tc_warps.cuh: the A operand's Philox noise drawn by the nt product kernel itself
struct FusePeer;    // tc_warps.cuh: the finished tiles of the tn product published for the exchange over the ranks

bool tc_available();

// ---- all-in-one entry points (split pre-pass + GEMM), used by mpvae_contract_nt / _tn ----
size_t tc_workspace_nt(int M, int N, int K);
size_t tc_workspace_tn(int M, int N1, int N2);
// C[M,N] = A[M,K] . B[N,K]^T
// reuse_planes != 0: skip the split pre-pass and use the operand planes a previous call left in `ws`
// (lets a caller time the GEMM kernel alone)
int tc_contract_nt(const float* A, const float* Bm, float* C, int M, int N, int K, void* ws, size_t ws_bytes,
                   cudaStream_t stream, int reuse_planes = 0, int exact = 0, int ldc = 0, int allow_ksplit = 0);
// C[N1,N2] = A[M,N1]^T . B[M,N2]
int tc_contract_tn(const float* A, const float* Bm, float* C, int M, int N1, int N2, void* ws, size_t ws_bytes,
                   cudaStream_t stream, int reuse_planes = 0, int exact = 0);

// ---- staged interface used by the probit forward / backward (operand planes persist between the two) ----
// An operand is stored as two planes [2][rows][pitch] (hi | lo) of fp16.  A row-major
// [rows][cols] operand serves both as a K-major operand of the nt product (cols = K) and as an MN-major operand of
// the tn product (rows = K): the noise planes written by the forward are reused by the backward as they are.
size_t tc_planes_bytes(int rows, int cols);
// absmax: device slot holding max|x| as fp32 bits (the pieces are scaled by 2^-exponent of it); nullptr = scale 1.
// compute_absmax != 0 runs the reduction first (slot must be zeroed by the caller).
// perm_S > 0: src rows are s-major (s * perm_B + b) and are written b-major (b * perm_S + s).
int tc_split(const float* src, int rows, int cols, void* planes, uint32_t* absmax, int compute_absmax, cudaStream_t stream,
             int src_pitch = 0, int perm_S = 0, int perm_B = 0);   // src_pitch: row pitch of src in floats (0 = cols)
// standard normals (Philox4x32-10, same stream of numbers as philox_normal_kernel) written directly as ONE plane whose
// rows are b-major: element (s, b, z) lands in row b * S + s
int tc_philox_planes(void* planes, int S, int B, int Z, int B_global, int row0, uint64_t seed, uint64_t offset,
                     const uint64_t* offset_dev, cudaStream_t stream);
// a_exact / b_exact: that operand lies exactly on the 11-bit piece grid and is stored as ONE plane (the library's own
// Philox noise): two MMA passes instead of three.
// Columns [N, ldc) of C are left alone unless write_pad != 0: then they are padding the caller owns, and the epilogue
// may fill them (with zeros) to store whole 16-byte vectors.
int tc_gemm_nt(const void* a_planes, const void* b_planes, float* C, int M, int N, int K, const uint32_t* absmax_a,
               const uint32_t* absmax_b, cudaStream_t stream, int ldc = 0, int a_exact = 0,   // ldc: pitch of C (0 = N)
               void* tail_scratch = nullptr, size_t tail_scratch_bytes = 0,
               const FuseNoise* noise = nullptr,    // noise != nullptr: a_planes is written by the kernel itself (a_exact)
               int write_pad = 0);
// tail_scratch (optional, tc_tail_scratch_bytes()): lets the kernel cut the tiles of the last, partial wave of its
// persistent grid into K-slices so that the wave does not leave most SMs idle.
size_t tc_tail_scratch_bytes();
int tc_pitch(int cols);                                      // plane row pitch (elements) for `cols` columns
int tc_absmax(const float* src, size_t n, uint32_t* out_bits, cudaStream_t stream);   // atomicMax of finite |x| bits into *out
int tc_gemm_tn(const void* a_planes, const void* b_planes, float* C, int M, int N1, int N2, const uint32_t* absmax_a,
               const uint32_t* absmax_b, cudaStream_t stream, int b_exact = 0, void* tail_scratch = nullptr,
               size_t tail_scratch_bytes = 0, int a_pitch = 0,
               // peer != nullptr: C is this rank's partial; the kernel PUBLISHES its finished tiles [0, *exchanged_tiles) in
               // per-tile counters in peer memory and leaves exchange_sms() SMs free for the exchange kernel the caller runs
               // beside it; the K-sliced tail tiles are left to the caller
               const FusePeer* peer = nullptr, int* exchanged_tiles = nullptr);
// SMs the g_R product leaves to the exchange kernel running beside it (even; MPVAE_EXCHANGE_SMS overrides: experiments)
int exchange_sms(int world);

}  // namespace mpv
