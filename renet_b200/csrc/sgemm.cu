// fp32 FFMA GEMMs used by the self-loop (RGCN.py:35) and the GRU projections (model.py:86,94).
// fp32 parity (1e-4 vs the CPU oracle) rules out single-pass TF32; these are plain FFMA kernels
// with register tiling.  The 3xTF32 tcgen05 path lives in umma_gemm.cu.
//
// Tile: 80 x 200 outputs per CTA (d_out = 200, 600 and 1200 are all multiples of 200, so no column
// waste), 8x8 outputs per thread, K stepped by 8 with register-staged double buffering.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace renet {

namespace {

constexpr int BM = 80, BN = 200, BK = 8;
constexpr int TX = 25, TY = 10;          // 250 compute threads (+6 that only help loading)
constexpr int NT = 256;
constexpr int BMP = BM + 4;              // padded leading dim of the transposed A tile

// C = A[idx] @ B (+bias) (+C)
template <bool INDEXED>
__global__ void __launch_bounds__(NT, 2)
sgemm_nn_kernel(const float* __restrict__ A, const int32_t* __restrict__ a_index, int64_t lda,
                const float* __restrict__ B, int64_t ldb, float* __restrict__ C, int64_t ldc,
                const float* __restrict__ bias, int64_t M, int N, int K, int accumulate) {
  __shared__ __align__(16) float As[2][BK][BMP];
  __shared__ __align__(16) float Bs[2][BK][BN];

  const int tid = threadIdx.x;
  const int tx = tid % TX, ty = tid / TX;
  const int64_t row0 = (int64_t)blockIdx.x * BM;
  const int col0 = blockIdx.y * BN;

  // ---- global -> register staging -------------------------------------------------------------
  const int a_row = tid >> 1, a_k4 = (tid & 1) * 4;      // tid < 160
  const bool a_active = tid < BM * BK / 4;
  const float* a_ptr = nullptr;
  if (a_active) {
    int64_t r = row0 + a_row;
    if (r < M) {
      int64_t rr = INDEXED ? (int64_t)__ldg(a_index + r) : r;
      a_ptr = A + rr * lda + a_k4;
    }
  }
  // B: 400 float4 per tile -> slots tid and tid+256
  const int b_k0 = tid / 50, b_n0 = (tid % 50) * 4;
  const int b_k1 = (tid + NT) / 50, b_n1 = ((tid + NT) % 50) * 4;
  const bool b1_active = (tid + NT) < BK * BN / 4;

  float4 a_reg = make_float4(0, 0, 0, 0), b_reg0 = a_reg, b_reg1 = a_reg;
  auto load_tile = [&](int k0) {
    a_reg = make_float4(0, 0, 0, 0);
    if (a_ptr != nullptr && k0 + a_k4 < K) a_reg = ldg_f4(a_ptr + k0);
    b_reg0 = make_float4(0, 0, 0, 0);
    if (k0 + b_k0 < K && col0 + b_n0 < N) b_reg0 = ldg_f4(B + (int64_t)(k0 + b_k0) * ldb + col0 + b_n0);
    b_reg1 = make_float4(0, 0, 0, 0);
    if (b1_active && k0 + b_k1 < K && col0 + b_n1 < N)
      b_reg1 = ldg_f4(B + (int64_t)(k0 + b_k1) * ldb + col0 + b_n1);
  };
  auto store_tile = [&](int buf) {
    if (a_active) {
      As[buf][a_k4 + 0][a_row] = a_reg.x;
      As[buf][a_k4 + 1][a_row] = a_reg.y;
      As[buf][a_k4 + 2][a_row] = a_reg.z;
      As[buf][a_k4 + 3][a_row] = a_reg.w;
    }
    st_f4(&Bs[buf][b_k0][b_n0], b_reg0);
    if (b1_active) st_f4(&Bs[buf][b_k1][b_n1], b_reg1);
  };

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  const int nk = (K + BK - 1) / BK;
  load_tile(0);
  store_tile(0);
  __syncthreads();
  for (int kt = 0; kt < nk; ++kt) {
    const int buf = kt & 1;
    if (kt + 1 < nk) load_tile((kt + 1) * BK);
    if (ty < TY) {
#pragma unroll
      for (int k = 0; k < BK; ++k) {
        // rows ty*4..+3 and 40+ty*4..+3 ; cols tx*4..+3 and 100+tx*4..+3 (conflict-free LDS.128)
        float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
        float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][40 + ty * 4]);
        float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
        float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][k][100 + tx * 4]);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
    }
    if (kt + 1 < nk) {
      store_tile(buf ^ 1);
      __syncthreads();
    }
  }

  if (ty >= TY) return;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t r = row0 + (i < 4 ? ty * 4 + i : 40 + ty * 4 + (i - 4));
    if (r >= M) continue;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int c = col0 + h * 100 + tx * 4;
      if (c >= N) continue;
      float4 v = make_float4(acc[i][h * 4 + 0], acc[i][h * 4 + 1], acc[i][h * 4 + 2], acc[i][h * 4 + 3]);
      if (bias != nullptr) {
        float4 bb = ldg_f4(bias + c);
        v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
      }
      float* cp = C + r * ldc + c;
      if (accumulate) {
        float4 o = *reinterpret_cast<const float4*>(cp);
        v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
      }
      st_f4(cp, v);
    }
  }
}

// Fallback for shapes the tiled kernel cannot take (K or N not a multiple of 4, unaligned): one
// thread per output.  Only tiny known-answer cases hit it.
__global__ void sgemm_nn_naive(const float* __restrict__ A, const int32_t* __restrict__ a_index, int64_t lda,
                               const float* __restrict__ B, int64_t ldb, float* __restrict__ C, int64_t ldc,
                               const float* __restrict__ bias, int64_t M, int N, int K, int accumulate) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * N) return;
  int64_t r = i / N;
  int c = (int)(i % N);
  int64_t rr = a_index ? (int64_t)a_index[r] : r;
  float s = 0.f;
  for (int k = 0; k < K; ++k) s = fmaf(A[rr * lda + k], B[(int64_t)k * ldb + c], s);
  if (bias) s += bias[c];
  if (accumulate) s += C[r * ldc + c];
  C[r * ldc + c] = s;
}

// ---- C[M,N] (+)= A^T B,  A [K, M] rows through a_index, B [K, N]; K is the long dimension ------
// Used for dWloop = Hin^T @ G (K = number of nodes).  Split-K over CTAs, fp32 atomics into C
// (C must be zero-initialised or hold the value to accumulate onto).
constexpr int TN_BM = 40, TN_BN = 200, TN_BK = 8, TN_KCHUNK = 256;
template <bool INDEXED>
__global__ void __launch_bounds__(256)
sgemm_tn_splitk_kernel(const float* __restrict__ A, const int32_t* __restrict__ a_index, int64_t lda,
                       const float* __restrict__ B, int64_t ldb, float* __restrict__ C, int64_t ldc,
                       int M, int N, int64_t K) {
  // tile: 40 (M) x 200 (N) outputs, thread = 4 x 8 outputs -> 10 x 25 threads
  __shared__ __align__(16) float As[TN_BK][TN_BM];
  __shared__ __align__(16) float Bs[TN_BK][TN_BN];
  const int tid = threadIdx.x;
  const int tx = tid % 25, ty = tid / 25;
  const int m0 = blockIdx.x * TN_BM, n0 = blockIdx.y * TN_BN;
  const int64_t kbeg = (int64_t)blockIdx.z * TN_KCHUNK;
  const int64_t kend = min(K, kbeg + TN_KCHUNK);
  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  for (int64_t k0 = kbeg; k0 < kend; k0 += TN_BK) {
    // A tile: 8 x 40 floats = 80 float4 ; B tile: 8 x 200 = 400 float4
    if (tid < 80) {
      int k = tid / 10, m4 = (tid % 10) * 4;
      float4 v = make_float4(0, 0, 0, 0);
      if (k0 + k < kend && m0 + m4 < M) {
        int64_t rr = INDEXED ? (int64_t)__ldg(a_index + k0 + k) : (k0 + k);
        v = ldg_f4(A + rr * lda + m0 + m4);
      }
      st_f4(&As[k][m4], v);
    }
    for (int i = tid; i < 400; i += 256) {
      int k = i / 50, n4 = (i % 50) * 4;
      float4 v = make_float4(0, 0, 0, 0);
      if (k0 + k < kend && n0 + n4 < N) v = ldg_f4(B + (k0 + k) * ldb + n0 + n4);
      st_f4(&Bs[k][n4], v);
    }
    __syncthreads();
    if (ty < 10) {
#pragma unroll
      for (int k = 0; k < TN_BK; ++k) {
        float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
        float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
        float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][100 + tx * 4]);
        const float a[4] = {a0.x, a0.y, a0.z, a0.w};
        const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
    }
    __syncthreads();
  }
  if (ty >= 10) return;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      int c = n0 + h * 100 + tx * 4;
      if (c >= N) continue;
      red_add_f4(C + (int64_t)m * ldc + c,
                 make_float4(acc[i][h * 4 + 0], acc[i][h * 4 + 1], acc[i][h * 4 + 2], acc[i][h * 4 + 3]));
    }
  }
}

__global__ void sgemm_tn_naive(const float* __restrict__ A, const int32_t* __restrict__ a_index, int64_t lda,
                               const float* __restrict__ B, int64_t ldb, float* __restrict__ C, int64_t ldc,
                               int M, int N, int64_t K) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * N) return;
  int m = i / N, n = i % N;
  float s = 0.f;
  for (int64_t k = 0; k < K; ++k) {
    int64_t rr = a_index ? (int64_t)a_index[k] : k;
    s = fmaf(A[rr * lda + m], B[k * ldb + n], s);
  }
  C[(int64_t)m * ldc + n] += s;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

int umma_gemm_nn_try(const float* A, const int32_t* a_index, int64_t lda, const float* B, int64_t ldb, float* C,
                     int64_t ldc, const float* bias, int64_t M, int32_t N, int32_t K, bool accumulate,
                     cudaStream_t stream);

// RENET_GEMM=ffma|umma selects the dense-GEMM engine (all are this library's own sm_100a kernels): 0 = FFMA, 1 = tensor
// cores (the self-loop shape on its persistent kernel); renet_set_gemm_engine(2) = tensor cores with the packed kernel for
// every shape (the previous self-loop kernel, kept for A/B comparisons).
static int g_gemm_mode = -1;
int gemm_mode() {
  if (g_gemm_mode < 0) {
    const char* e = getenv("RENET_GEMM");
    g_gemm_mode = (e != nullptr && strcmp(e, "ffma") == 0) ? 0 : 1;   // default: tensor cores
  }
  return g_gemm_mode;
}
int set_gemm_mode(int m) {
  const int prev = gemm_mode();
  g_gemm_mode = m == 2 ? 2 : (m ? 1 : 0);
  return prev;
}

int sgemm_nn(const float* A, const int32_t* a_index, int64_t lda, const float* B, int64_t ldb, float* C,
             int64_t ldc, const float* bias, int64_t M, int32_t N, int32_t K, bool accumulate,
             cudaStream_t stream) {
  if (M <= 0 || N <= 0) return RENET_OK;
  if (gemm_mode() != 0) {   // tcgen05 3xTF32 path (umma_gemm.cu); returns 0 when the shape is not supported
    const int r = umma_gemm_nn_try(A, a_index, lda, B, ldb, C, ldc, bias, M, N, K, accumulate, stream);
    if (r != 0) return r < 0 ? r : RENET_OK;
  }
  const bool fast = (K % 4 == 0) && (N % 4 == 0) && (lda % 4 == 0) && (ldb % 4 == 0) && (ldc % 4 == 0) &&
                    aligned16(A) && aligned16(B) && aligned16(C) && (bias == nullptr || aligned16(bias));
  if (fast) {
    dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)((N + BN - 1) / BN));
    if (a_index)
      sgemm_nn_kernel<true><<<grid, NT, 0, stream>>>(A, a_index, lda, B, ldb, C, ldc, bias, M, N, K, accumulate);
    else
      sgemm_nn_kernel<false><<<grid, NT, 0, stream>>>(A, a_index, lda, B, ldb, C, ldc, bias, M, N, K, accumulate);
    RENET_CHECK_LAUNCH("sgemm_nn_kernel");
  } else {
    int64_t total = M * N;
    sgemm_nn_naive<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(A, a_index, lda, B, ldb, C, ldc, bias, M,
                                                                       N, K, accumulate);
    RENET_CHECK_LAUNCH("sgemm_nn_naive");
  }
  return RENET_OK;
}

int sgemm_tn(const float* A, const int32_t* a_index, int64_t lda, const float* B, int64_t ldb, float* C,
             int64_t ldc, int32_t M, int32_t N, int64_t K, bool accumulate, cudaStream_t stream) {
  if (M <= 0 || N <= 0) return RENET_OK;
  if (!accumulate) RENET_CHECK_CUDA(cudaMemset2DAsync(C, ldc * sizeof(float), 0, N * sizeof(float), M, stream));
  if (K <= 0) return RENET_OK;
  const bool fast = (M % 4 == 0) && (N % 4 == 0) && (lda % 4 == 0) && (ldb % 4 == 0) && (ldc % 4 == 0) &&
                    aligned16(A) && aligned16(B) && aligned16(C);
  if (fast) {
    dim3 grid((M + TN_BM - 1) / TN_BM, (N + TN_BN - 1) / TN_BN, (unsigned)((K + TN_KCHUNK - 1) / TN_KCHUNK));
    if (a_index)
      sgemm_tn_splitk_kernel<true><<<grid, 256, 0, stream>>>(A, a_index, lda, B, ldb, C, ldc, M, N, K);
    else
      sgemm_tn_splitk_kernel<false><<<grid, 256, 0, stream>>>(A, a_index, lda, B, ldb, C, ldc, M, N, K);
    RENET_CHECK_LAUNCH("sgemm_tn_splitk_kernel");
  } else {
    sgemm_tn_naive<<<(M * N + 255) / 256, 256, 0, stream>>>(A, a_index, lda, B, ldb, C, ldc, M, N, K);
    RENET_CHECK_LAUNCH("sgemm_tn_naive");
  }
  return RENET_OK;
}

}  // namespace renet
