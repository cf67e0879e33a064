// fp32-accurate GEMM on the 5th-generation tensor cores: C[M,N] = A[M,K] @ B[K,N] (+bias) (+C)
//
// RE-Net's dense work on the hot path -- the self-loop H @ W_loop (RGCN.py:35) and the GRU input /
// recurrent projections (model.py:86,94) -- must match a CPU fp32 oracle to 1e-4, which single-pass
// TF32 (10-bit mantissa, ~3e-4 on K=200) does not.  This kernel issues tcgen05.mma kind::tf32 with the
// 3xTF32 split:  a = a_hi + a_lo,  b = b_hi + b_lo  (hi = top 19 bits, lo = a - a_hi exactly),
//     D += a_hi*b_hi + a_lo*b_hi + a_hi*b_lo        (fp32 accumulation in TMEM)
// which recovers ~fp32 accuracy (dropped term a_lo*b_lo ~ 2^-22 relative) at 1/3 of TF32 peak -- still
// several times the FFMA roofline.
//
// Structure (one CTA per 128-row tile of A x one <=200-column tile of B, 256 threads):
//   * operands are staged by the threads themselves (not TMA): A rows may be gathered through an index
//     (fused embedding lookup / read-out), B is row-major [K,N] and has to be transposed to K-major,
//     and both need the hi/lo split, so a register pass is required anyway;
//   * smem holds two stages of {A_hi, A_lo [128 x 40], B_hi, B_lo [208 x 40]} in the canonical
//     no-swizzle K-major UMMA layout (8-row x 16-byte core matrices; LBO = one 4-column slab,
//     SBO = 128 B);
//   * one elected thread issues 15 MMAs (5 k-steps x 3 split products, M=128, N=208, K=8) per stage and
//     commits to an mbarrier that frees the stage; loads of chunk c+1 overlap the MMAs of chunk c;
//   * accumulator: 128 lanes x 208 fp32 columns of TMEM (256 allocated); epilogue reads it with
//     tcgen05.ld 32x32b (thread = row) and writes C with bias / accumulate applied.
#include "common.cuh"
#include <mutex>
#include <vector>

#include "umma.cuh"

namespace renet {
namespace {

constexpr int UM = 128;          // rows per CTA tile
constexpr int UN = 200;          // logical columns per CTA tile
constexpr int UNP = 208;         // padded to a multiple of 16 for the MMA N
constexpr int UKC = 40;          // K per stage (5 MMA k-steps of 8)
constexpr int USLABS = UKC / 4;  // 16-byte (4 x fp32) column slabs per stage
constexpr int UTHREADS = 256;
constexpr int A_SLAB_BYTES = UM * 16;    // 2048
constexpr int B_SLAB_BYTES = UNP * 16;   // 3328
constexpr int A_BYTES = USLABS * A_SLAB_BYTES;   // 20480
constexpr int B_BYTES = USLABS * B_SLAB_BYTES;   // 33280
constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;   // 107520
constexpr int NUM_STAGES = 2;
constexpr int SMEM_BYTES = NUM_STAGES * STAGE_BYTES + 64;   // + mbarriers / tmem pointer
constexpr int TMEM_COLS = 256;

__device__ __forceinline__ uint32_t make_idesc() { return make_idesc_n(UNP); }

template <bool INDEXED>
__global__ void __launch_bounds__(UTHREADS, 1)
umma_gemm_nn_kernel(const float* __restrict__ A, const int32_t* __restrict__ a_index, int64_t lda,
                    const float* __restrict__ B, int64_t ldb, float* __restrict__ C, int64_t ldc,
                    const float* __restrict__ bias, int64_t M, int N, int K, int accumulate) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t row0 = (int64_t)blockIdx.x * UM;
  const int n0 = blockIdx.y * UN;
  const int tile_n = min(UN, N - n0);

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NUM_STAGES * STAGE_BYTES);   // [0..1] stage free, [2] done
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + NUM_STAGES * STAGE_BYTES + 32);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar0 = smem_u32(bars);

  if (tid == 0) {
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    mbar_init(bar0 + 16, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // zero the 8 padding rows (n = 200..207) of every B slab once; they are never written again
  for (int i = tid; i < NUM_STAGES * 2 * USLABS * (UNP - UN); i += UTHREADS) {
    const int r = i % (UNP - UN), sl = (i / (UNP - UN)) % USLABS, which = (i / ((UNP - UN) * USLABS)) % 2,
              st = i / ((UNP - UN) * USLABS * 2);
    float4* p = reinterpret_cast<float4*>(smem + st * STAGE_BYTES + 2 * A_BYTES + which * B_BYTES + sl * B_SLAB_BYTES +
                                          (UN + r) * 16);
    *p = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t idesc = make_idesc();

  // per-thread A source rows: task = slab * 128 + row  (5 tasks per thread per chunk)
  const float* a_rows[5];
#pragma unroll
  for (int t = 0; t < 5; ++t) {
    const int task = tid + t * UTHREADS;
    const int r = task % UM;
    const int64_t gr = row0 + r;
    a_rows[t] = nullptr;
    if (gr < M) {
      const int64_t rr = INDEXED ? (int64_t)__ldg(a_index + gr) : gr;
      a_rows[t] = A + rr * lda;
    }
  }

  const int nchunks = K / UKC;
  for (int c = 0; c < nchunks; ++c) {
    const int st = c % NUM_STAGES;
    uint8_t* sA_hi = smem + st * STAGE_BYTES;
    uint8_t* sA_lo = sA_hi + A_BYTES;
    uint8_t* sB_hi = sA_lo + A_BYTES;
    uint8_t* sB_lo = sB_hi + B_BYTES;
    if (c >= NUM_STAGES) mbar_wait(bar0 + 8 * st, ((c / NUM_STAGES) - 1) & 1);   // MMAs of chunk c-2 done
    const int k0 = c * UKC;
    // ---- A: 128 rows x 10 slabs; thread -> (slab, row): conflict-free 16-byte smem stores ----------
#pragma unroll
    for (int t = 0; t < 5; ++t) {
      const int task = tid + t * UTHREADS;
      const int sl = task / UM, r = task % UM;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a_rows[t] != nullptr) v = ldg_f4(a_rows[t] + k0 + 4 * sl);
      float4 hi, lo;
      split4(v, hi, lo);
      *reinterpret_cast<float4*>(sA_hi + sl * A_SLAB_BYTES + r * 16) = hi;
      *reinterpret_cast<float4*>(sA_lo + sl * A_SLAB_BYTES + r * 16) = lo;
    }
    // ---- B: [40 k] x [200 n] row-major -> K-major: 4x4 register transposes -----------------------------
    for (int task = tid; task < USLABS * (UN / 4); task += UTHREADS) {
      const int sl = task / (UN / 4), j = task % (UN / 4);
      float4 m[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        m[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (4 * j < tile_n) m[i] = ldg_f4(B + (int64_t)(k0 + 4 * sl + i) * ldb + n0 + 4 * j);
      }
      const float4 t0 = make_float4(m[0].x, m[1].x, m[2].x, m[3].x);
      const float4 t1 = make_float4(m[0].y, m[1].y, m[2].y, m[3].y);
      const float4 t2 = make_float4(m[0].z, m[1].z, m[2].z, m[3].z);
      const float4 t3 = make_float4(m[0].w, m[1].w, m[2].w, m[3].w);
      const float4 tr[4] = {t0, t1, t2, t3};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float4 hi, lo;
        split4(tr[q], hi, lo);
        *reinterpret_cast<float4*>(sB_hi + sl * B_SLAB_BYTES + (4 * j + q) * 16) = hi;
        *reinterpret_cast<float4*>(sB_lo + sl * B_SLAB_BYTES + (4 * j + q) * 16) = lo;
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> async proxy (MMA)
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t a_hi = smem_base + st * STAGE_BYTES, a_lo = a_hi + A_BYTES;
      const uint32_t b_hi = a_lo + A_BYTES, b_lo = b_hi + B_BYTES;
#pragma unroll
      for (int ks = 0; ks < UKC / 8; ++ks) {
        const uint32_t ao = ks * 2 * A_SLAB_BYTES, bo = ks * 2 * B_SLAB_BYTES;
        const uint64_t dAh = make_desc(a_hi + ao, A_SLAB_BYTES, 128), dAl = make_desc(a_lo + ao, A_SLAB_BYTES, 128);
        const uint64_t dBh = make_desc(b_hi + bo, B_SLAB_BYTES, 128), dBl = make_desc(b_lo + bo, B_SLAB_BYTES, 128);
        umma_tf32(tmem_base, dAh, dBh, idesc, (c | ks) != 0);
        umma_tf32(tmem_base, dAl, dBh, idesc, 1);
        umma_tf32(tmem_base, dAh, dBl, idesc, 1);
      }
      umma_commit(bar0 + 8 * st);                         // frees this stage when the MMAs have read it
      if (c == nchunks - 1) umma_commit(bar0 + 16);       // accumulator complete
    }
  }

  // ---- epilogue: TMEM -> registers -> global (thread = row; warps 0-3 cols [0,104), warps 4-7 [104,208)) ---
  mbar_wait(bar0 + 16, 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  {
    const int q = warp & 3, half = warp >> 2;
    const int r = q * 32 + lane;
    const int64_t gr = row0 + r;
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
    for (int cc = half * 104; cc < half * 104 + 104; cc += 8) {
      uint32_t v[8];
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                   : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                   : "r"(taddr + (uint32_t)cc));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (gr < M && cc < tile_n) {
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = __uint_as_float(v[i]);
        float* cp = C + gr * ldc + n0 + cc;
        if (bias != nullptr) {
          const float4 b0 = ldg_f4(bias + n0 + cc), b1 = ldg_f4(bias + n0 + cc + 4);
          o[0] += b0.x; o[1] += b0.y; o[2] += b0.z; o[3] += b0.w;
          o[4] += b1.x; o[5] += b1.y; o[6] += b1.z; o[7] += b1.w;
        }
        if (accumulate) {
          const float4 c0 = *reinterpret_cast<const float4*>(cp), c1 = *reinterpret_cast<const float4*>(cp + 4);
          o[0] += c0.x; o[1] += c0.y; o[2] += c0.z; o[3] += c0.w;
          o[4] += c1.x; o[5] += c1.y; o[6] += c1.z; o[7] += c1.w;
        }
        st_f4(cp, make_float4(o[0], o[1], o[2], o[3]));
        st_f4(cp + 4, make_float4(o[4], o[5], o[6], o[7]));
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
  }
}


// ======================================================================================================
// v2: pre-packed B + TMA bulk copies + 128-byte swizzle
//
// Profiling v1 showed the tile time dominated by operand staging, not by the MMAs: every CTA re-transposed and
// re-split the same B (W_loop / GRU weights), and the no-swizzle layout forced row-strided A loads (16 useful
// bytes per 128-byte line with almost no L1 left beside 215 KB of shared memory).  v2:
//   * B is packed ONCE per GEMM by umma_pack_b_kernel into the exact shared-memory image (hi and lo planes,
//     K-major, SWIZZLE_128B, one 53 KB block per (column tile, 32-wide K chunk)); the GEMM CTAs fetch a block
//     with a single cp.async.bulk (TMA) that completes on the stage's mbarrier;
//   * A is staged by the threads with fully coalesced 128-byte row segments and conflict-free swizzled
//     16-byte stores (chunk j of row r lands at chunk j ^ (r % 8));
//   * K is processed in chunks of 32 (one swizzle atom): 4 MMA k-steps x 3 split products per chunk.
// ======================================================================================================
constexpr int P_BK = 32;
constexpr int P_A_BYTES = UM * 128;                  // 16384
constexpr int P_B_BYTES = UNP * 128;                 // 26624
constexpr int P_B_CHUNK = 2 * P_B_BYTES;             // hi + lo planes of one (tile, chunk)
constexpr int P_SMEM = 4 * P_A_BYTES + 2 * P_B_CHUNK + 1024 + 128;   // two tiles' A (hi,lo) + two B stages

// Bp[(nt * n_chunks + kc)] = {hi plane, lo plane} of B[kc*32 .. +31][nt*200 .. +207] (zero padded)
__global__ void __launch_bounds__(256)
umma_pack_b_kernel(const float* __restrict__ B, int64_t sk, int64_t sn, int N, int K, uint8_t* __restrict__ Bp,
                   int n_chunks, int tile_offset) {
  // logical B[k][n] = B[k*sk + n*sn]  (row-major [K,N]: sk = ldb, sn = 1; a [N,K] weight read transposed: sk = 1, sn = ld)
  const int nt = blockIdx.x, kc = blockIdx.y;
  const int n0 = nt * UN, k0 = kc * P_BK;
  const int tile_n = min(UN, N - n0);
  uint8_t* dst = Bp + (size_t)((nt + tile_offset) * n_chunks + kc) * P_B_CHUNK;
  for (int task = blockIdx.z * 256 + threadIdx.x; task < UNP * 8; task += 256 * gridDim.z) {
    const int j = task / UNP, n = task % UNP;      // consecutive threads -> consecutive n (coalesced reads)
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = k0 + 4 * j + i;
      v[i] = (n < tile_n && k < K) ? __ldg(B + (int64_t)k * sk + (int64_t)(n0 + n) * sn) : 0.f;
    }
    float4 hi, lo;
    split4(make_float4(v[0], v[1], v[2], v[3]), hi, lo);
    const uint32_t off = sw128_offset(n, j);
    *reinterpret_cast<float4*>(dst + off) = hi;
    *reinterpret_cast<float4*>(dst + P_B_BYTES + off) = lo;
  }
}

// Fused-epilogue modes of the packed kernel (the decoder of model.py:89-91,97-100: logits = X @ W^T + b, cross-entropy):
//   EPI 0  C = acc (+bias) (+C)                                   -- plain GEMM
//   EPI 1  per (row, half column tile): running max and sum of exp of the logits, and the target's logit -- the
//          [M, N] logits never reach memory; ce_reduce_kernel turns the partials into logsumexp and the loss
//   EPI 2  dlogits[row, col] = (exp(logit - lse[row]) - [col == target[row]]) * scale, written to memory for the two
//          gradient GEMMs (the backward pass recomputes the logits instead of keeping them)

// One CTA = a PAIR of 128-row tiles sharing every B block: the packed B chunk (53 KB) is fetched once per pair,
// the two tiles' A buffers ping-pong (tile 1's chunk is staged while tile 0's MMAs run and vice versa), and the
// two accumulators live side by side in TMEM (2 x 256 columns).
template <bool INDEXED, int EPI = 0>
__global__ void __launch_bounds__(UTHREADS, 1)
umma_gemm_packed_kernel(const float* __restrict__ A, const int32_t* __restrict__ a_index, int64_t lda,
                        const uint8_t* __restrict__ Bp, float* __restrict__ C, int64_t ldc,
                        const float* __restrict__ bias, int64_t M, int N, int K, int n_chunks, int accumulate,
                        int64_t batch_a, int64_t batch_bp, int64_t batch_c, EpiArgs epi, int k_splits, int64_t split_c) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024 - (raw & 1023)) & 1023);     // swizzle atoms need 1024-byte alignment
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // grid.z = batch x K-split.  Batched GEMMs (the two GRU encoders): per-batch operand offsets.  Split-K (long-K,
  // few-tile products such as dX = dlogits @ W of the decoder): split s owns the chunks [s*cps, (s+1)*cps) and writes its
  // partial product to C + s*split_c; the caller sums the partials.
  const int zb = blockIdx.z / k_splits, split = blockIdx.z - zb * k_splits;
  A += zb * batch_a;
  Bp += zb * batch_bp;
  C += zb * batch_c + (int64_t)split * split_c;
  if (bias != nullptr) bias += zb * (int64_t)N;
  const int cps = (n_chunks + k_splits - 1) / k_splits;
  const int c_begin = split * cps;
  const int n_local = min(cps, n_chunks - c_begin);      // >= 1: the launcher never creates an empty split
  const int64_t row_base = (int64_t)blockIdx.x * (2 * UM);
  const int nt = blockIdx.y;
  const int n0 = nt * UN;
  const int tile_n = min(UN, N - n0);
  // smem: A[2 tiles][hi,lo] (4 x 16 KB), B[2 stages][hi,lo] (2 x 53 KB), barriers
  uint8_t* sA = smem;
  uint8_t* sB = smem + 4 * P_A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + 2 * P_B_CHUNK);   // [0,1] B landed, [2,3] B free, [4,5] A_t free, [6] done
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar0 = smem_u32(bars);
  if (tid == 0) {
    for (int i = 0; i < 7; ++i) mbar_init(bar0 + 8 * i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t idesc = make_idesc();

  // A tasks per tile: 128 rows x 8 sixteen-byte chunks = 1024 -> 4 per thread; 8 consecutive lanes read one
  // 128-byte row segment (coalesced), and write it to 8 distinct swizzled chunks (conflict-free)
  const float* a_rows[2][4];
  uint32_t a_off[4];
  int a_k[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int task = tid + t * UTHREADS;
    const int r = task >> 3, j = task & 7;
    a_off[t] = sw128_offset(r, j);
    a_k[t] = 4 * j;
#pragma unroll
    for (int tl = 0; tl < 2; ++tl) {
      const int64_t gr = row_base + tl * UM + r;
      a_rows[tl][t] = nullptr;
      if (gr < M) {
        const int64_t rr = INDEXED ? (int64_t)__ldg(a_index + gr) : gr;
        a_rows[tl][t] = A + rr * lda;
      }
    }
  }
  const uint8_t* bp_tile = Bp + (size_t)nt * n_chunks * P_B_CHUNK;
  float4 vnext[4];
  auto load_a = [&](int tl, int c) {
    const int k0 = (c_begin + c) * P_BK;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      vnext[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a_rows[tl][t] != nullptr && k0 + a_k[t] < K) vnext[t] = ldg_f4(a_rows[tl][t] + k0 + a_k[t]);
    }
  };
  load_a(0, 0);
  for (int c = 0; c < n_local; ++c) {
    const int bs = c & 1;
    if (tid == 0) {   // TMA: one bulk copy per chunk brings the packed B block for BOTH tiles
      if (c >= 2) mbar_wait(bar0 + 16 + 8 * bs, ((c >> 1) - 1) & 1);          // both tiles' MMAs of chunk c-2 done
      const uint32_t full = bar0 + 8 * bs;
      const uint32_t dstB = smem_base + 4 * P_A_BYTES + bs * P_B_CHUNK;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "r"((uint32_t)P_B_CHUNK) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dstB),
                   "l"(bp_tile + (size_t)(c_begin + c) * P_B_CHUNK), "r"((uint32_t)P_B_CHUNK), "r"(full)
                   : "memory");
    }
#pragma unroll
    for (int tl = 0; tl < 2; ++tl) {
      uint8_t* sA_hi = sA + tl * 2 * P_A_BYTES;
      uint8_t* sA_lo = sA_hi + P_A_BYTES;
      if (c >= 1) mbar_wait(bar0 + 32 + 8 * tl, (c - 1) & 1);                 // MMAs of (tile tl, chunk c-1) have read A_tl
      float4 v[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) v[t] = vnext[t];
      if (tl == 0) load_a(1, c);                                              // next step's global loads fly during this step
      else if (c + 1 < n_local) load_a(0, c + 1);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float4 hi, lo;
        split4(v[t], hi, lo);
        *reinterpret_cast<float4*>(sA_hi + a_off[t]) = hi;
        *reinterpret_cast<float4*>(sA_lo + a_off[t]) = lo;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();
      if (tid == 0) {
        if (tl == 0) mbar_wait(bar0 + 8 * bs, (c >> 1) & 1);                  // B block landed
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a_hi = smem_base + tl * 2 * P_A_BYTES, a_lo = a_hi + P_A_BYTES;
        const uint32_t b_hi = smem_base + 4 * P_A_BYTES + bs * P_B_CHUNK, b_lo = b_hi + P_B_BYTES;
        const uint32_t acc = tmem_base + tl * 256;
#pragma unroll
        for (int ks = 0; ks < P_BK / 8; ++ks) {
          const uint32_t ko = ks * 32;                       // 8 fp32 = 32 bytes along the swizzled row
          const uint64_t dAh = make_desc_sw128(a_hi + ko), dAl = make_desc_sw128(a_lo + ko);
          const uint64_t dBh = make_desc_sw128(b_hi + ko), dBl = make_desc_sw128(b_lo + ko);
          umma_tf32(acc, dAh, dBh, idesc, (c | ks) != 0);
          umma_tf32(acc, dAl, dBh, idesc, 1);
          umma_tf32(acc, dAh, dBl, idesc, 1);
        }
        umma_commit(bar0 + 32 + 8 * tl);                     // A_tl may be overwritten
        if (tl == 1) {
          umma_commit(bar0 + 16 + 8 * bs);                   // B stage may be overwritten
          if (c == n_local - 1) umma_commit(bar0 + 48);      // both accumulators complete
        }
      }
    }
  }

  mbar_wait(bar0 + 48, 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  {
    // thread = accumulator row; warps 0-3 take columns [0,104), warps 4-7 [104,208): 3 x (32 columns) + 1 x 8
    const int q = warp & 3, half = warp >> 2;
    const int r = q * 32 + lane;
    const int cbase = half * 104;
#pragma unroll 1
    for (int tl = 0; tl < 2; ++tl) {
      const int64_t gr = row_base + tl * UM + r;
      const uint32_t taddr = tmem_base + tl * 256 + ((uint32_t)(q * 32) << 16);
      // EPI 1 state of this thread's (row, half tile): running max / sum of exp; EPI 2: the row's logsumexp and target
      float run_m = -3.0e38f, run_s = 0.f;
      const int tgt = (EPI != 0 && gr < M) ? __ldg(epi.target + gr) : -1;
      const float row_lse = (EPI == 2 && gr < M) ? __ldg(epi.lse + gr) : 0.f;
      const float gscale = (EPI == 2) ? epi.scale * (epi.dscale != nullptr ? __ldg(epi.dscale) : 1.f) : 0.f;
      auto emit8 = [&](const uint32_t* v8, int cc) {
        if (gr < M && cc < tile_n) {
          float o[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) o[i] = __uint_as_float(v8[i]);
          if (EPI != 0) {
            // fused cross-entropy epilogues: columns are guarded one by one (the class count need not be a multiple of 8)
            const int nv = min(8, tile_n - cc);
            float mx = -3.0e38f;
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (i < nv) {
                if (bias != nullptr) o[i] += __ldg(bias + n0 + cc + i);
                mx = fmaxf(mx, o[i]);
              }
            if (EPI == 1) {
              const float nm = fmaxf(run_m, mx);
              float add = 0.f;
#pragma unroll
              for (int i = 0; i < 8; ++i)
                if (i < nv) {
                  add += expf(o[i] - nm);
                  if (n0 + cc + i == tgt) epi.tlogit[gr] = o[i];
                }
              run_s = run_s * expf(run_m - nm) + add;
              run_m = nm;
            } else {
              float* dp = C + gr * ldc + n0 + cc;
#pragma unroll
              for (int i = 0; i < 8; ++i)
                if (i < nv) {
                  const float gv = (expf(o[i] - row_lse) - (n0 + cc + i == tgt ? 1.f : 0.f)) * gscale;
                  dp[i] = gv;                                              // row-major: A of dX = dlogits @ W
                  epi.dT[(int64_t)(n0 + cc + i) * epi.ldT + gr] = gv;      // transposed (lanes = consecutive rows: coalesced)
                }
            }
            return;
          }
          float* cp = C + gr * ldc + n0 + cc;
          if (bias != nullptr) {
            const float4 b0 = ldg_f4(bias + n0 + cc), b1 = ldg_f4(bias + n0 + cc + 4);
            o[0] += b0.x; o[1] += b0.y; o[2] += b0.z; o[3] += b0.w;
            o[4] += b1.x; o[5] += b1.y; o[6] += b1.z; o[7] += b1.w;
          }
          if (accumulate) {
            const float4 c0 = *reinterpret_cast<const float4*>(cp), c1 = *reinterpret_cast<const float4*>(cp + 4);
            o[0] += c0.x; o[1] += c0.y; o[2] += c0.z; o[3] += c0.w;
            o[4] += c1.x; o[5] += c1.y; o[6] += c1.z; o[7] += c1.w;
          }
          st_f4(cp, make_float4(o[0], o[1], o[2], o[3]));
          st_f4(cp + 4, make_float4(o[4], o[5], o[6], o[7]));
        }
      };
#pragma unroll 1
      for (int blk = 0; blk < 3; ++blk) {
        uint32_t v[32];
        const int cc = cbase + blk * 32;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
              "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
              "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
              "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(taddr + (uint32_t)cc));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int g8 = 0; g8 < 4; ++g8) emit8(v + 8 * g8, cc + 8 * g8);
      }
      {
        uint32_t v8[8];
        const int cc = cbase + 96;
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(v8[0]), "=r"(v8[1]), "=r"(v8[2]), "=r"(v8[3]), "=r"(v8[4]), "=r"(v8[5]), "=r"(v8[6]), "=r"(v8[7])
                     : "r"(taddr + (uint32_t)cc));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        emit8(v8, cc);
      }
      if (EPI == 1 && gr < M) {
        const int64_t pi = (int64_t)(nt * 2 + half) * M + gr;
        epi.pmax[pi] = run_m;
        epi.psum[pi] = run_s;
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
  }
}

// ======================================================================================================
// v3: the self-loop product C[M, 200] = A[idx[m]] @ W_loop (N = 200, one packed column tile; no bias, no accumulate)
//
// The packed kernel runs stage-A / MMA rounds separated by CTA-wide barriers followed by a serial epilogue, and gives
// every CTA 256 rows: a layer-2 shape (S ~ 8.5k rows) occupies 34 of 148 SMs.  This kernel is persistent and
// warp-specialised:
//   * grid = min(units, SMs); CTA b owns units b, b + grid, b + 2 grid, ... (at most ceil(units / grid) each);
//   * a unit is 128 rows x all 208 columns; when the row tiles fill at most half of the SMs, a unit is 128 rows x one
//     column half instead: N = 112 (columns 0..111) or N = 96 (112..207).  Both are legal M = 128 MMA widths and both
//     start on a 1024-byte swizzle atom of the packed image (row 112 = 14 KB), so TMA fetches just that half's rows;
//   * roles, all hand-offs on mbarriers (no CTA-wide barrier in the main loop):
//       warps 0-7    gather the A rows through the index, split hi/lo, store them swizzled into a 3-stage ring;
//       warp 8       (one lane) streams the packed B chunks with cp.async.bulk into a 2-stage ring;
//       warp 9       (one lane) issues the MMAs and commits; it also owns the TMEM allocation;
//       warps 10-13  drain the accumulators (warp w reads TMEM lanes 32 (w % 4) ..);
//   * two TMEM accumulators (columns [0, 256) and [256, 512)): unit i's epilogue overlaps unit i+1's MMAs;
//   * the last K chunk issues only the k-steps that carry data (1 of 4 for K = 200).  The products keep the packed
//     kernel's order (per k-step hi.hi, lo.hi, hi.lo; k ascending): the skipped k-steps only added zeros;
//   * epilogue: tcgen05.ld of 32 rows x 32 columns -> a per-warp padded shared tile -> 128-byte row segments to C.
// Shared memory (bytes): A ring 3 x 32768 + B ring 2 x 53248 + epilogue 4 x 4608 + barriers 128 + alignment 1024
// = 224384 (219 KB of the 227 KB a block may have).
constexpr int SL_PROD_WARPS = 8;
constexpr int SL_PROD = SL_PROD_WARPS * 32;
constexpr int SL_TMA_WARP = 8;
constexpr int SL_MMA_WARP = 9;
constexpr int SL_EPI_WARP0 = 10;
constexpr int SL_THREADS = (SL_EPI_WARP0 + 4) * 32;      // 448
constexpr int SL_A_STAGES = 3;
constexpr int SL_B_STAGES = 2;
constexpr int SL_A_STAGE = 2 * P_A_BYTES;                 // hi + lo planes of 128 rows x 32 k
constexpr int SL_EPI_LD = 36;                             // floats per staged row: 32 + 4 keeps 16-byte accesses conflict-free
constexpr int SL_EPI_WARP_BYTES = 32 * SL_EPI_LD * 4;     // 4608
constexpr int SL_OFF_B = SL_A_STAGES * SL_A_STAGE;
constexpr int SL_OFF_EPI = SL_OFF_B + SL_B_STAGES * P_B_CHUNK;
constexpr int SL_OFF_BAR = SL_OFF_EPI + 4 * SL_EPI_WARP_BYTES;
constexpr int SL_SMEM = SL_OFF_BAR + 128 + 1024;
constexpr int SL_HALF0_N = 112;                           // width of the first column half; the second is UNP - 112 = 96
static_assert(SL_SMEM <= 227 * 1024, "self-loop kernel: shared memory budget");
static_assert((SL_HALF0_N * 128) % 1024 == 0, "column half must start on a swizzle atom");
// mbarrier slots (8 bytes each) after SL_OFF_BAR
constexpr int SL_BAR_A_FULL = 0, SL_BAR_A_EMPTY = 3, SL_BAR_B_FULL = 6, SL_BAR_B_EMPTY = 8, SL_BAR_T_FULL = 10,
              SL_BAR_T_EMPTY = 12, SL_NUM_BARS = 14;

struct SlUnit {
  int64_t row0;   // first row of the 128-row tile
  int col0;       // first accumulator column within the 208-column tile
  int n;          // MMA width: 208, 112 or 96
};
__device__ __forceinline__ SlUnit sl_unit(int u, int split) {
  SlUnit s;
  if (split) {
    s.row0 = (int64_t)(u >> 1) * UM;
    s.col0 = (u & 1) ? SL_HALF0_N : 0;
    s.n = (u & 1) ? UNP - SL_HALF0_N : SL_HALF0_N;
  } else {
    s.row0 = (int64_t)u * UM;
    s.col0 = 0;
    s.n = UNP;
  }
  return s;
}

template <bool INDEXED>
__global__ void __launch_bounds__(SL_THREADS, 1)
umma_selfloop_kernel(const float* __restrict__ A, const int32_t* __restrict__ a_index, int64_t lda,
                     const uint8_t* __restrict__ Bp, float* __restrict__ C, int64_t ldc, int64_t M, int K, int n_chunks,
                     int n_units, int split) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024 - (raw & 1023)) & 1023);     // swizzle atoms need 1024-byte alignment
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar0 = smem_base + SL_OFF_BAR;
  auto bar = [&](int i) { return bar0 + 8 * i; };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SL_OFF_BAR + 8 * SL_NUM_BARS);

  if (tid == 0) {
    for (int s = 0; s < SL_A_STAGES; ++s) {
      mbar_init(bar(SL_BAR_A_FULL + s), SL_PROD);
      mbar_init(bar(SL_BAR_A_EMPTY + s), 1);
    }
    for (int s = 0; s < SL_B_STAGES; ++s) {
      mbar_init(bar(SL_BAR_B_FULL + s), 1);
      mbar_init(bar(SL_BAR_B_EMPTY + s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar(SL_BAR_T_FULL + a), 1);
      mbar_init(bar(SL_BAR_T_EMPTY + a), 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == SL_MMA_WARP) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  const int n_local = (n_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // >= 1: grid <= n_units
  const int total = n_local * n_chunks;                                                  // (unit, K chunk) items
  const int last_ks = (K - (n_chunks - 1) * P_BK + 7) / 8;                              // k-steps of the last chunk

  if (warp < SL_PROD_WARPS) {
    // ---- A producers: 128 rows x 8 sixteen-byte chunks per K chunk = 4 tasks per thread; 8 consecutive lanes read one
    // 128-byte row segment (coalesced) and write 8 distinct swizzled chunks (conflict-free).  The global loads of item
    // it+1 are issued before item it is stored, and before waiting for its stage to be free.
    const int j = tid & 7;
    uint32_t a_off[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) a_off[t] = sw128_offset((tid >> 3) + 32 * t, j);
    const float* rows[4];
    float4 vnext[4];
    auto set_rows = [&](int lu) {
      const SlUnit un = sl_unit((int)blockIdx.x + lu * (int)gridDim.x, split);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int64_t gr = un.row0 + (tid >> 3) + 32 * t;
        rows[t] = nullptr;
        if (gr < M) rows[t] = A + (INDEXED ? (int64_t)__ldg(a_index + gr) : gr) * lda;
      }
    };
    auto load = [&](int c) {
      const int k = c * P_BK + 4 * j;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        vnext[t] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rows[t] != nullptr && k < K) vnext[t] = ldg_f4(rows[t] + k);
      }
    };
    set_rows(0);
    load(0);
    for (int it = 0; it < total; ++it) {
      const int s = it % SL_A_STAGES, round = it / SL_A_STAGES;
      float4 v[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) v[t] = vnext[t];
      if (it + 1 < total) {
        const int lu = (it + 1) / n_chunks, c = it + 1 - lu * n_chunks;
        if (c == 0) set_rows(lu);
        load(c);
      }
      if (round > 0) mbar_wait(bar(SL_BAR_A_EMPTY + s), (round - 1) & 1);   // the MMAs of item it-3 have read the stage
      uint8_t* sA_hi = smem + s * SL_A_STAGE;
      uint8_t* sA_lo = sA_hi + P_A_BYTES;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float4 hi, lo;
        split4(v[t], hi, lo);
        *reinterpret_cast<float4*>(sA_hi + a_off[t]) = hi;
        *reinterpret_cast<float4*>(sA_lo + a_off[t]) = lo;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");         // generic-proxy writes -> async proxy (MMA)
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(SL_BAR_A_FULL + s)) : "memory");
    }
  } else if (warp == SL_TMA_WARP) {
    if (lane == 0) {
      // ---- B: one (unit, chunk) item = the chunk's packed block, or the rows of the unit's column half of it --------
      for (int it = 0; it < total; ++it) {
        const int s = it % SL_B_STAGES, round = it / SL_B_STAGES;
        const int lu = it / n_chunks, c = it - lu * n_chunks;
        const SlUnit un = sl_unit((int)blockIdx.x + lu * (int)gridDim.x, split);
        if (round > 0) mbar_wait(bar(SL_BAR_B_EMPTY + s), (round - 1) & 1);
        const uint32_t full = bar(SL_BAR_B_FULL + s);
        const uint32_t dst = smem_base + SL_OFF_B + s * P_B_CHUNK;
        const uint8_t* src = Bp + (size_t)c * P_B_CHUNK + un.col0 * 128;
        const uint32_t plane = (uint32_t)un.n * 128;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "r"(2 * plane) : "memory");
        if (un.n == UNP) {      // full width: the hi and lo planes are contiguous
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                       "l"(src), "r"((uint32_t)P_B_CHUNK), "r"(full)
                       : "memory");
        } else {
#pragma unroll
          for (int p = 0; p < 2; ++p)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             dst + p * P_B_BYTES),
                         "l"(src + p * P_B_BYTES), "r"(plane), "r"(full)
                         : "memory");
        }
      }
    }
    __syncwarp();
  } else if (warp == SL_MMA_WARP) {
    if (lane == 0) {
      int it = 0;
      for (int lu = 0; lu < n_local; ++lu) {
        const int acc = lu & 1;
        const SlUnit un = sl_unit((int)blockIdx.x + lu * (int)gridDim.x, split);
        const uint32_t idesc = make_idesc_n(un.n);
        if (lu >= 2) mbar_wait(bar(SL_BAR_T_EMPTY + acc), ((lu >> 1) - 1) & 1);   // epilogue of unit lu-2 has drained it
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d = tmem_base + acc * 256;
        for (int c = 0; c < n_chunks; ++c, ++it) {
          const int sa = it % SL_A_STAGES, sb = it % SL_B_STAGES;
          mbar_wait(bar(SL_BAR_A_FULL + sa), (it / SL_A_STAGES) & 1);
          mbar_wait(bar(SL_BAR_B_FULL + sb), (it / SL_B_STAGES) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t a_hi = smem_base + sa * SL_A_STAGE, a_lo = a_hi + P_A_BYTES;
          const uint32_t b_hi = smem_base + SL_OFF_B + sb * P_B_CHUNK, b_lo = b_hi + P_B_BYTES;
          const int nks = (c == n_chunks - 1) ? last_ks : P_BK / 8;
          for (int ks = 0; ks < nks; ++ks) {
            const uint32_t ko = ks * 32;                       // 8 fp32 = 32 bytes along the swizzled row
            const uint64_t dAh = make_desc_sw128(a_hi + ko), dAl = make_desc_sw128(a_lo + ko);
            const uint64_t dBh = make_desc_sw128(b_hi + ko), dBl = make_desc_sw128(b_lo + ko);
            umma_tf32(d, dAh, dBh, idesc, (c | ks) != 0);
            umma_tf32(d, dAl, dBh, idesc, 1);
            umma_tf32(d, dAh, dBl, idesc, 1);
          }
          umma_commit(bar(SL_BAR_A_EMPTY + sa));               // both stages may be overwritten once these MMAs are done
          umma_commit(bar(SL_BAR_B_EMPTY + sb));
        }
        umma_commit(bar(SL_BAR_T_FULL + acc));                 // accumulator complete
      }
    }
    __syncwarp();
  } else {
    // ---- epilogue: TMEM -> registers (thread = row, 32 columns) -> padded shared tile -> 8 lanes per 128-byte row segment
    const int q = warp & 3;
    float* stg = reinterpret_cast<float*>(smem + SL_OFF_EPI + (warp - SL_EPI_WARP0) * SL_EPI_WARP_BYTES);
    for (int lu = 0; lu < n_local; ++lu) {
      const int acc = lu & 1;
      const SlUnit un = sl_unit((int)blockIdx.x + lu * (int)gridDim.x, split);
      const int col_end = min(UN, un.col0 + un.n);
      const int nblk = (un.n + 31) / 32;
      mbar_wait(bar(SL_BAR_T_FULL + acc), (lu >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t taddr = tmem_base + acc * 256 + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int blk = 0; blk < nblk; ++blk) {
        uint32_t v[32];
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
              "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
              "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
              "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(taddr + (uint32_t)(blk * 32)));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (blk == nblk - 1) {     // every column of this accumulator is in registers: the MMAs may reuse it
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(SL_BAR_T_EMPTY + acc)) : "memory");
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
          *reinterpret_cast<uint4*>(stg + lane * SL_EPI_LD + 4 * i) = make_uint4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        __syncwarp();
#pragma unroll
        for (int p = 0; p < 8; ++p) {
          const int r = 4 * p + (lane >> 3), c4 = lane & 7;
          const int64_t gr = un.row0 + q * 32 + r;
          const int gc = un.col0 + blk * 32 + 4 * c4;
          if (gr < M && gc < col_end) st_f4(C + gr * ldc + gc, *reinterpret_cast<const float4*>(stg + r * SL_EPI_LD + 4 * c4));
        }
        __syncwarp();
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == SL_MMA_WARP) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
  }
}

}  // namespace

// Returns 1 if the shape was taken by the tensor-core path (launch enqueued), 0 if the caller should
// fall back to the FFMA kernel, negative on error.
static uint8_t* g_scratch = nullptr;
static int64_t g_scratch_bytes = 0;
void set_scratch(void* p, int64_t bytes) { g_scratch = (uint8_t*)p; g_scratch_bytes = p ? bytes : 0; }

// ---- packed-weight cache (renet_set_weight_generation) ------------------------------------------------------------------
// Packing a weight into the UMMA operand image is a kernel launch per weight per call.  Weights only change when the
// optimiser steps, so the caller may declare a "weight generation": while it is unchanged, a packed image made for a
// given (device, pointers, shape) key is valid and reused; a new generation invalidates every image (the buffers are
// kept and overwritten by the next pack).  generation < 0 (the default) turns the cache off.
namespace {
struct PackEntry {
  int device;
  const void* keys[6];
  int nkeys;
  int64_t bytes;
  void* buf;
  int64_t gen;
};
std::mutex g_pack_mu;
std::vector<PackEntry> g_pack_entries;
int64_t g_weight_generation = -1;
}  // namespace

void set_weight_generation(int64_t g) {
  std::lock_guard<std::mutex> lk(g_pack_mu);
  g_weight_generation = g;
}

void* packed_cache_lookup(const void* const* keys, int nkeys, int64_t bytes, bool* hit) {
  *hit = false;
  std::lock_guard<std::mutex> lk(g_pack_mu);
  if (g_weight_generation < 0 || nkeys > 6) return nullptr;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  for (auto& e : g_pack_entries) {
    if (e.device != dev || e.nkeys != nkeys || e.bytes != bytes) continue;
    bool same = true;
    for (int i = 0; i < nkeys; ++i) same &= e.keys[i] == keys[i];
    if (!same) continue;
    *hit = e.gen == g_weight_generation;
    e.gen = g_weight_generation;
    return e.buf;
  }
  if (g_pack_entries.size() >= 64) {       // bounded: drop the oldest image
    cudaFree(g_pack_entries.front().buf);
    g_pack_entries.erase(g_pack_entries.begin());
  }
  PackEntry e{};
  e.device = dev; e.nkeys = nkeys; e.bytes = bytes; e.gen = g_weight_generation;
  for (int i = 0; i < nkeys; ++i) e.keys[i] = keys[i];
  if (cudaMalloc(&e.buf, (size_t)bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  g_pack_entries.push_back(e);
  return e.buf;
}

// ---- building blocks shared with gru.cu ------------------------------------------------------------------------
int64_t umma_packed_bytes(int N, int K) {
  return (int64_t)((N + UN - 1) / UN) * ((K + P_BK - 1) / P_BK) * P_B_CHUNK;
}
bool umma_shape_ok(int N, int K) { return (K % 4 == 0) && (N % 8 == 0) && N > 0 && K > 0; }

// Pack logical B[k][n] = B[k*sk + n*sn] (K x N) into tiles [tile_offset, tile_offset + ceil(N/200)) of Bp.
int umma_pack_b(const float* B, int64_t sk, int64_t sn, int N, int K, void* Bp, int tile_offset, cudaStream_t stream) {
  const int n_tiles = (N + UN - 1) / UN, n_chunks = (K + P_BK - 1) / P_BK;
  umma_pack_b_kernel<<<dim3(n_tiles, n_chunks, 7), 256, 0, stream>>>(B, sk, sn, N, K, (uint8_t*)Bp, n_chunks, tile_offset);
  RENET_CHECK_LAUNCH("umma_pack_b_kernel");
  return RENET_OK;
}

// C[b] (+)= A[b] @ Bpacked[b] (+bias[b]) for b < batch; strides in elements (A, C) / bytes (Bp).
// epi_mode 1 / 2: fused cross-entropy epilogues (EpiArgs); k_splits > 1: split-K partial products at C + s*split_c.
int umma_gemm_prepacked_ex(const float* A, const int32_t* a_index, int64_t lda, const void* Bp, float* C, int64_t ldc,
                           const float* bias, int64_t M, int N, int K, bool accumulate, int batch, int64_t batch_a,
                           int64_t batch_bp, int64_t batch_c, int epi_mode, const EpiArgs& epi, int k_splits, int64_t split_c,
                           cudaStream_t stream) {
  if (M <= 0) return RENET_OK;
  static bool attr2 = false;
  if (!attr2) {
    RENET_CHECK_CUDA(cudaFuncSetAttribute(umma_gemm_packed_kernel<true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM));
    RENET_CHECK_CUDA(cudaFuncSetAttribute(umma_gemm_packed_kernel<false, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM));
    RENET_CHECK_CUDA(cudaFuncSetAttribute(umma_gemm_packed_kernel<false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM));
    RENET_CHECK_CUDA(cudaFuncSetAttribute(umma_gemm_packed_kernel<false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM));
    attr2 = true;
  }
  const int n_tiles = (N + UN - 1) / UN, n_chunks = (K + P_BK - 1) / P_BK;
  if (k_splits < 1) k_splits = 1;
  if (k_splits > n_chunks) k_splits = n_chunks;
  while (k_splits > 1 && ((n_chunks + k_splits - 1) / k_splits) * (k_splits - 1) >= n_chunks) --k_splits;   // no empty split
  dim3 grid((unsigned)((M + 2 * UM - 1) / (2 * UM)), (unsigned)n_tiles, (unsigned)(batch * k_splits));
#define RENET_UMMA_LAUNCH(IDX, EP)                                                                                       \
  umma_gemm_packed_kernel<IDX, EP><<<grid, UTHREADS, P_SMEM, stream>>>(A, a_index, lda, (const uint8_t*)Bp, C, ldc, bias, M, N, K, \
                                                                      n_chunks, accumulate, batch_a, batch_bp, batch_c, epi,  \
                                                                      k_splits, split_c)
  if (epi_mode == 1) RENET_UMMA_LAUNCH(false, 1);
  else if (epi_mode == 2) RENET_UMMA_LAUNCH(false, 2);
  else if (a_index) RENET_UMMA_LAUNCH(true, 0);
  else RENET_UMMA_LAUNCH(false, 0);
#undef RENET_UMMA_LAUNCH
  RENET_CHECK_LAUNCH("umma_gemm_packed_kernel");
  return k_splits;      // > 0: the number of K-splits actually used (1 = C holds the result)
}

int umma_gemm_prepacked(const float* A, const int32_t* a_index, int64_t lda, const void* Bp, float* C, int64_t ldc,
                        const float* bias, int64_t M, int N, int K, bool accumulate, int batch, int64_t batch_a,
                        int64_t batch_bp, int64_t batch_c, cudaStream_t stream) {
  EpiArgs none{};
  const int r = umma_gemm_prepacked_ex(A, a_index, lda, Bp, C, ldc, bias, M, N, K, accumulate, batch, batch_a, batch_bp, batch_c,
                                       0, none, 1, 0, stream);
  return r < 0 ? r : RENET_OK;
}

// C[M, 200] = A[(a_index)] @ Bpacked with the persistent self-loop kernel (v3 above).
static int umma_selfloop(const float* A, const int32_t* a_index, int64_t lda, const void* Bp, float* C, int64_t ldc,
                         int64_t M, int K, cudaStream_t stream) {
  static bool attr = false;
  if (!attr) {
    RENET_CHECK_CUDA(cudaFuncSetAttribute(umma_selfloop_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SL_SMEM));
    RENET_CHECK_CUDA(cudaFuncSetAttribute(umma_selfloop_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SL_SMEM));
    attr = true;
  }
  static int sm_count[64] = {0};
  int dev = 0;
  RENET_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) dev = 0;
  if (sm_count[dev] == 0) RENET_CHECK_CUDA(cudaDeviceGetAttribute(&sm_count[dev], cudaDevAttrMultiProcessorCount, dev));
  const int sms = sm_count[dev];
  const int64_t tiles = (M + UM - 1) / UM;
  // Column halves double the units (and read every A row twice); they pay off only while the whole-width units leave
  // at least half of the SMs idle.
  const int split = 2 * tiles <= sms ? 1 : 0;
  const int64_t units = split ? 2 * tiles : tiles;
  RENET_CHECK_ARG(units < (int64_t)1 << 30, "umma_selfloop: too many rows");
  const int grid = (int)(units < sms ? units : sms);
  const int n_chunks = (K + P_BK - 1) / P_BK;
  if (a_index)
    umma_selfloop_kernel<true><<<grid, SL_THREADS, SL_SMEM, stream>>>(A, a_index, lda, (const uint8_t*)Bp, C, ldc, M, K,
                                                                     n_chunks, (int)units, split);
  else
    umma_selfloop_kernel<false><<<grid, SL_THREADS, SL_SMEM, stream>>>(A, a_index, lda, (const uint8_t*)Bp, C, ldc, M, K,
                                                                      n_chunks, (int)units, split);
  RENET_CHECK_LAUNCH("umma_selfloop_kernel");
  return RENET_OK;
}

int umma_gemm_nn_try(const float* A, const int32_t* a_index, int64_t lda, const float* B, int64_t ldb, float* C,
                     int64_t ldc, const float* bias, int64_t M, int32_t N, int32_t K, bool accumulate,
                     cudaStream_t stream) {
  const bool aligned = ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B) | reinterpret_cast<uintptr_t>(C) |
                         reinterpret_cast<uintptr_t>(bias)) & 15) == 0;
  // ---- packed path: needs the registered scratch buffer for the packed copy of B ---------------------------------
  if (aligned && umma_shape_ok(N, K) && (lda % 4 == 0) && (ldc % 4 == 0) && M >= 64 && g_scratch != nullptr &&
      umma_packed_bytes(N, K) <= g_scratch_bytes && (reinterpret_cast<uintptr_t>(g_scratch) & 127) == 0) {
    bool hit = false;
    const void* keys[4] = {B, reinterpret_cast<const void*>((intptr_t)ldb), reinterpret_cast<const void*>((intptr_t)N),
                           reinterpret_cast<const void*>((intptr_t)K)};
    void* cached = packed_cache_lookup(keys, 4, umma_packed_bytes(N, K), &hit);
    void* Bp = cached ? cached : g_scratch;
    int rc = hit ? 0 : umma_pack_b(B, ldb, 1, N, K, Bp, 0, stream);
    if (rc) return rc;
    // the self-loop shape (H @ W_loop, RGCN.py:35) takes the persistent kernel unless engine 2 asks for the packed one
    if (gemm_mode() == 1 && N == UN && K == UN && bias == nullptr && !accumulate)
      rc = umma_selfloop(A, a_index, lda, Bp, C, ldc, M, K, stream);
    else
      rc = umma_gemm_prepacked(A, a_index, lda, Bp, C, ldc, bias, M, N, K, accumulate, 1, 0, 0, 0, stream);
    return rc ? rc : 1;
  }
  const bool ok = (K % UKC == 0) && K >= UKC && (N % 8 == 0) && (lda % 4 == 0) && (ldb % 4 == 0) && (ldc % 4 == 0) &&
                  M >= 64 && aligned;
  if (!ok) return 0;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e1 = cudaFuncSetAttribute(umma_gemm_nn_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    cudaError_t e2 = cudaFuncSetAttribute(umma_gemm_nn_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e1 != cudaSuccess || e2 != cudaSuccess) {
      set_error("cudaFuncSetAttribute(umma_gemm_nn_kernel) failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
      return RENET_ERR_CUDA;
    }
    attr_set = true;
  }
  dim3 grid((unsigned)((M + UM - 1) / UM), (unsigned)((N + UN - 1) / UN));
  if (a_index)
    umma_gemm_nn_kernel<true><<<grid, UTHREADS, SMEM_BYTES, stream>>>(A, a_index, lda, B, ldb, C, ldc, bias, M, N, K, accumulate);
  else
    umma_gemm_nn_kernel<false><<<grid, UTHREADS, SMEM_BYTES, stream>>>(A, a_index, lda, B, ldb, C, ldc, bias, M, N, K, accumulate);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("launch of umma_gemm_nn_kernel failed: %s", cudaGetErrorString(e));
    return RENET_ERR_CUDA;
  }
  count_launch();
  return 1;
}

}  // namespace renet
