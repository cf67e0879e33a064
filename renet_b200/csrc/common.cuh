// Shared helpers for librenet_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/renet_b200.h"

namespace renet {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define RENET_CHECK_ARG(cond, ...)                  \
  do {                                              \
    if (!(cond)) {                                  \
      ::renet::set_error(__VA_ARGS__);              \
      return RENET_ERR_INVALID_ARG;                 \
    }                                               \
  } while (0)

#define RENET_CHECK_CUDA(expr)                                                        \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      ::renet::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),     \
                         __FILE__, __LINE__);                                         \
      return RENET_ERR_CUDA;                                                          \
    }                                                                                 \
  } while (0)

#define RENET_CHECK_LAUNCH(name)                                                      \
  do {                                                                                \
    cudaError_t _e = cudaGetLastError();                                              \
    if (_e != cudaSuccess) {                                                          \
      ::renet::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));    \
      return RENET_ERR_CUDA;                                                          \
    }                                                                                 \
    ::renet::count_launch();                                                          \
  } while (0)

constexpr int kNumSMs = 148;  // B200

__device__ __forceinline__ float4 ldg_f4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
// streaming 128-bit load that does not allocate in L1 (keeps L1 for the relation-weight table)
__device__ __forceinline__ float4 ldg_f4_stream(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_f4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// 128-bit vector reduction to global memory (sm_90+): one RED for four floats.
__device__ __forceinline__ void red_add_f4(float* p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

// internal (non-exported) launchers shared between translation units -------------------------------
// C[M,N] (ldc) = A[M,K] (rows optionally through a_index; lda) @ B[K,N] (ldb) [+ bias[N]] [+ C if accumulate]
int sgemm_nn(const float* A, const int32_t* a_index, int64_t lda, const float* B, int64_t ldb, float* C,
             int64_t ldc, const float* bias, int64_t M, int32_t N, int32_t K, bool accumulate,
             cudaStream_t stream);
// C[M,N] += / = A^T B with A [K,M] (rows of A optionally through a_index), B [K,N]:  C = A^T @ B
int sgemm_tn(const float* A, const int32_t* a_index, int64_t lda, const float* B, int64_t ldb, float* C,
             int64_t ldc, int32_t M, int32_t N, int64_t K, bool accumulate, cudaStream_t stream);
// C[M,N] = A[M,K] @ B^T with B [N,K]
int sgemm_nt(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
             int64_t M, int32_t N, int32_t K, bool accumulate, cudaStream_t stream);

// 0 = automatic, 1 = tile, 3 = stream (RENET_GATHER_KERNEL=tile|stream; rgcn_fwd.cu)
int gather_kernel_choice();
constexpr int64_t kStreamMinEdges = 16384;   // below this a persistent 148-CTA launch costs more than the tile kernel
constexpr int64_t kStreamMinNodes = 16384;
constexpr int64_t kStreamMaxNodes = 98304;    // 79 MB of fp32 features: beyond this the source rows come from HBM, not L2
bool gather_use_stream(int64_t E, int64_t N);
void set_stream_debug_buffer(long long* p);   // debug: per-warp time stamps of the stream kernel (rgcn_fwd.cu)          // the stream kernel (rgcn_stream.cuh) serves this edge count

// tcgen05 GEMM engine building blocks (umma_gemm.cu); gemm_mode() != 0 selects the engine (2: no persistent self-loop kernel)
int gemm_mode();
int64_t umma_packed_bytes(int N, int K);
// packed-weight cache (umma_gemm.cu): persistent device buffer for this key, or nullptr when caching is off; *hit says
// whether it already holds the image for the current weight generation
void set_weight_generation(int64_t g);
void* packed_cache_lookup(const void* const* keys, int nkeys, int64_t bytes, bool* hit);
bool umma_shape_ok(int N, int K);
int umma_pack_b(const float* B, int64_t sk, int64_t sn, int N, int K, void* Bp, int tile_offset, cudaStream_t stream);
// fused epilogues of the packed tcgen05 GEMM (umma_gemm.cu): see the comment there
struct EpiArgs {
  const int32_t* target;   // [M] class of every row
  const float* lse;        // [M] (EPI 2)
  float* pmax;             // [2 * n_tiles, M] (EPI 1)
  float* psum;             // [2 * n_tiles, M] (EPI 1)
  float* tlogit;           // [M] (EPI 1): written by the one thread that sees the target column
  float* dT;               // [N, ldT] (EPI 2): the same gradient transposed (A operand of dW = dlogits^T @ X)
  int64_t ldT;
  float scale;             // (EPI 2)
  const float* dscale;     // (EPI 2) optional device scalar multiplied into scale (the upstream gradient, no host read)
};
int umma_gemm_prepacked_ex(const float* A, const int32_t* a_index, int64_t lda, const void* Bp, float* C, int64_t ldc,
                           const float* bias, int64_t M, int N, int K, bool accumulate, int batch, int64_t batch_a,
                           int64_t batch_bp, int64_t batch_c, int epi_mode, const EpiArgs& epi, int k_splits, int64_t split_c,
                           cudaStream_t stream);
int umma_gemm_prepacked(const float* A, const int32_t* a_index, int64_t lda, const void* Bp, float* C, int64_t ldc,
                        const float* bias, int64_t M, int N, int K, bool accumulate, int batch, int64_t batch_a,
                        int64_t batch_bp, int64_t batch_c, cudaStream_t stream);

}  // namespace renet
