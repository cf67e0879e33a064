// Read-out + concat + GRU (reference Aggregator.py:139-165, model.py:86,94).
//
// The reference materialises zero-padded [Q,10,4h] / [Q,10,3h] inputs with a Python loop of 2Q
// cat/repeat/index_put launches ("# Slow!!!", Aggregator.py:148-155) and hands them to cuDNN.
// Here the concat never exists: W_ih . x is split column-wise into
//     GI[row]  = H2[readout[row]] @ Wrow           (per read-out row, S x h  @ h x 6h)
//     PQ[q]    = ent[s_q] @ Went + rel[r_q] @ Wrel + b_ih   (once per sequence)
//     PT[t]    = glob[t] @ Wglob                   (once per distinct timestamp)
// for both encoders at once (they share H2 rows, ent and glob), and every time step is one
// recurrent GEMM + one fused gate kernel over the sequences still active at that step.
#include "common.cuh"

namespace renet {
namespace {

// dst[k, dst_off + o] = src[o, src_off + k]   for o < rows_src, k < h
__global__ void pack_transpose_kernel(const float* __restrict__ src, int ld_src, int src_off, int rows_src,
                                      float* __restrict__ dst, int ld_dst, int dst_off, int h) {
  __shared__ float tile[32][33];
  const int o0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    int o = o0 + i, k = k0 + tx;
    tile[i][tx] = (o < rows_src && k < h) ? src[(int64_t)o * ld_src + src_off + k] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    int k = k0 + i, o = o0 + tx;
    if (o < rows_src && k < h) dst[(int64_t)k * ld_dst + dst_off + o] = tile[tx][i];
  }
}

__global__ void concat_bias_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out,
                                   int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i];
  else if (i < 2 * n) out[i] = b[i - n];
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// One GRU time step for both encoders.  Thread = (sequence q < n_act, encoder, unit).
//   gi = GI[row] + PQ[q] + PT[row_glob[row]]   (b_ih already folded into PQ)
//   gh = GH[q] + b_hh                           (GH = h_prev @ W_hh^T, or absent at t = 0)
__global__ void gru_gate_kernel(const float* __restrict__ GI, const float* __restrict__ PQ,
                                const float* __restrict__ PT, const float* __restrict__ GH,
                                const float* __restrict__ bhh /* [6h] */, const int32_t* __restrict__ row_glob,
                                const int32_t* __restrict__ seq_start, const int32_t* __restrict__ seq_len,
                                const float* __restrict__ Hprev /* [Q,2h] or null (t=0) */,
                                float* __restrict__ Hnext /* [Q,2h] */, float* __restrict__ hn4,
                                float* __restrict__ hn3, int n_act, int h, int t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int per_q = 2 * h;
  if (i >= n_act * per_q) return;
  const int q = i / per_q, c = i % per_q;
  const int enc = c / h, u = c % h;
  const int64_t row = (int64_t)seq_start[q] + t;
  const int64_t g = (int64_t)row_glob[row];
  const int base = enc * 3 * h + u;
  const float* gi = GI + row * 6 * h + base;
  const float* pq = PQ + (int64_t)q * 6 * h + base;
  const float* pt = PT + g * 6 * h + base;
  const float i_r = gi[0] + pq[0] + pt[0];
  const float i_z = gi[h] + pq[h] + pt[h];
  const float i_n = gi[2 * h] + pq[2 * h] + pt[2 * h];
  float h_r = bhh[base], h_z = bhh[base + h], h_n = bhh[base + 2 * h], hp = 0.f;
  if (Hprev != nullptr) {
    const float* gh = GH + (int64_t)q * 6 * h + base;
    h_r += gh[0]; h_z += gh[h]; h_n += gh[2 * h];
    hp = Hprev[(int64_t)q * per_q + c];
  }
  const float r = sigmoidf_(i_r + h_r);
  const float z = sigmoidf_(i_z + h_z);
  const float n = tanhf(i_n + r * h_n);
  const float hv = (1.f - z) * n + z * hp;
  Hnext[(int64_t)q * per_q + c] = hv;
  if (t == seq_len[q] - 1) (enc == 0 ? hn4 : hn3)[(int64_t)q * h + u] = hv;
}

// Packed (time-major) GRU inputs exactly as the reference aggregator returns them.
__global__ void pack_inputs_kernel(const float* __restrict__ H2, const int32_t* __restrict__ readout,
                                   const int32_t* __restrict__ row_glob, const float* __restrict__ glob,
                                   const float* __restrict__ ent, const float* __restrict__ rel,
                                   const int32_t* __restrict__ row_seq, const int32_t* __restrict__ seq_s,
                                   const int32_t* __restrict__ seq_r, const int32_t* __restrict__ packed_row,
                                   float* __restrict__ X4, float* __restrict__ X3, int64_t S, int h) {
  const int64_t p = blockIdx.x;  // packed position
  if (p >= S) return;
  const int64_t row = packed_row[p];
  const int q = row_seq[row];
  const float* a = H2 + (int64_t)readout[row] * h;
  const float* b = ent + (int64_t)seq_s[q] * h;
  const float* c = rel + (int64_t)seq_r[q] * h;
  const float* d = glob + (int64_t)row_glob[row] * h;
  float* x4 = X4 + p * 4 * h;
  float* x3 = X3 + p * 3 * h;
  for (int i = threadIdx.x; i < h; i += blockDim.x) {
    const float va = a[i], vb = b[i], vc = c[i], vd = d[i];
    x4[i] = va; x4[h + i] = vb; x4[2 * h + i] = vc; x4[3 * h + i] = vd;
    x3[i] = va; x3[h + i] = vb; x3[2 * h + i] = vd;
  }
}


// ---- input dropout (Aggregator.py:157-158) -----------------------------------------------------------------------------------
// The reference drops elements of the padded GRU inputs [Q,10,4h] and [Q,10,3h] independently (two nn.Dropout calls).
// With dropout the column-wise split of W_ih.x no longer applies (ent[s], rel[r], glob[t] get a different mask at every
// step), so the masked inputs are materialised once (sequence-major rows, S x 4h and S x 3h) and projected by two
// tensor-core GEMMs; the recurrence kernel is unchanged.  Masks come from Philox4x32-10 keyed by (seed, element index):
// nothing is stored, the backward pass regenerates them.
__device__ __forceinline__ uint4 philox4x32_10(uint64_t ctr, uint64_t key) {
  uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0u, c3 = 0u;
  uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
// keep-scale of element idx: 0 (dropped, probability p) or 1/(1-p)
__device__ __forceinline__ float dropout_scale(uint64_t idx, uint64_t seed, float p, float inv_keep) {
  const uint4 r = philox4x32_10(idx >> 2, seed);
  const uint32_t w = (idx & 3) == 0 ? r.x : ((idx & 3) == 1 ? r.y : ((idx & 3) == 2 ? r.z : r.w));
  return (w * 2.3283064365386963e-10f) >= p ? inv_keep : 0.f;
}

__global__ void dropout_mask_kernel(uint64_t seed, uint64_t offset, int64_t n, float p, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = dropout_scale(offset + (uint64_t)i, seed, p, 1.f / (1.f - p));
}

// masked inputs, sequence-major: row i = (sequence row_seq[i], its step i - seq_start[q])
__global__ void pack_inputs_dropout_kernel(const float* __restrict__ H2, const int32_t* __restrict__ readout,
                                           const int32_t* __restrict__ row_glob, const float* __restrict__ glob,
                                           const float* __restrict__ ent, const float* __restrict__ rel,
                                           const int32_t* __restrict__ row_seq, const int32_t* __restrict__ seq_s,
                                           const int32_t* __restrict__ seq_r, float* __restrict__ X4,
                                           float* __restrict__ X3, int64_t S, int h, float p, uint64_t seed) {
  const int64_t row = blockIdx.x;
  if (row >= S) return;
  const int q = row_seq[row];
  const float* src[4] = {H2 + (int64_t)readout[row] * h, ent + (int64_t)seq_s[q] * h, rel + (int64_t)seq_r[q] * h,
                         glob + (int64_t)row_glob[row] * h};
  const float inv = 1.f / (1.f - p);
  const uint64_t base4 = (uint64_t)row * 4 * h, base3 = (uint64_t)S * 4 * h + (uint64_t)row * 3 * h;
  for (int c = threadIdx.x; c < 4 * h; c += blockDim.x) {
    const int part = c / h, k = c - part * h;
    const float v = src[part][k];
    X4[row * 4 * h + c] = v * dropout_scale(base4 + c, seed, p, inv);
    if (part != 2) {                                   // X3 = [row | ent | glob]
      const int c3 = (part == 3 ? 2 * h : part * h) + k;
      X3[row * 3 * h + c3] = v * dropout_scale(base3 + c3, seed, p, inv);
    }
  }
}

// backward of the above: masked input gradients scattered to H2 rows / ent / rel / glob
__global__ void unpack_inputs_dropout_kernel(const float* __restrict__ dX4, const float* __restrict__ dX3,
                                             const int32_t* __restrict__ readout, const int32_t* __restrict__ row_glob,
                                             const int32_t* __restrict__ row_seq, const int32_t* __restrict__ seq_s,
                                             const int32_t* __restrict__ seq_r, float* __restrict__ dH2,
                                             float* __restrict__ d_ent, float* __restrict__ d_rel, float* __restrict__ d_glob,
                                             int64_t S, int h, float p, uint64_t seed) {
  const int64_t row = blockIdx.x;
  if (row >= S) return;
  const int q = row_seq[row];
  float* dst[4] = {dH2 + (int64_t)readout[row] * h, d_ent + (int64_t)seq_s[q] * h, d_rel + (int64_t)seq_r[q] * h,
                   d_glob != nullptr ? d_glob + (int64_t)row_glob[row] * h : nullptr};
  const float inv = 1.f / (1.f - p);
  const uint64_t base4 = (uint64_t)row * 4 * h, base3 = (uint64_t)S * 4 * h + (uint64_t)row * 3 * h;
  for (int c = threadIdx.x; c < 4 * h; c += blockDim.x) {
    const int part = c / h, k = c - part * h;
    float gsum = dX4[row * 4 * h + c] * dropout_scale(base4 + c, seed, p, inv);
    if (part != 2) {
      const int c3 = (part == 3 ? 2 * h : part * h) + k;
      gsum += dX3[row * 3 * h + c3] * dropout_scale(base3 + c3, seed, p, inv);
    }
    if (dst[part] != nullptr && gsum != 0.f) atomicAdd(dst[part] + k, gsum);
  }
}

// PQ[q, :] = b_ih (both encoders) for every sequence
__global__ void fill_rows_kernel(const float* __restrict__ v, float* __restrict__ out, int64_t rows, int cols) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows * cols) out[i] = v[i % cols];
}

struct GruWs {
  float *Brow, *Bent, *Brel, *Bglob, *Whh, *bih, *bhh, *GI, *PQ, *PT, *GH, *Hs;
  float *P_row, *P_ent, *P_rel, *P_glob, *P_hh;   // tensor-core engine: weights packed for umma_gemm_prepacked
  float *Xd4, *Xd3, *P_x4, *P_x3, *zrow;            // input-dropout / dense path: masked inputs [S,4h] / [S,3h], packed W_ih, S zero ints
  float* sync;                                      // grid-barrier counter of the persistent recurrence kernel
  int64_t p_hh_bytes;
  int64_t total_floats;
};

inline int64_t align4(int64_t x) { return (x + 3) & ~int64_t(3); }

GruWs carve(float* base, int64_t S, int64_t Q, int64_t T, int h, int max_len, bool dropout = false) {
  GruWs w;
  int64_t off = 0;
  auto take = [&](int64_t n) { float* p = base ? base + off : nullptr; off += align4(n); return p; };
  w.Brow = take((int64_t)h * 6 * h);
  w.Bent = take((int64_t)h * 6 * h);
  w.Brel = take((int64_t)h * 3 * h);
  w.Bglob = take((int64_t)h * 6 * h);
  w.Whh = take((int64_t)h * 6 * h);
  w.bih = take(6 * h);
  w.bhh = take(6 * h);
  w.GI = take(S * 6 * h);
  w.PQ = take(Q * 6 * h);
  w.PT = take(T * 6 * h);
  w.GH = take((int64_t)max_len * Q * 6 * h);   // recurrent pre-activations of every step (kept for backward)
  w.Hs = take((int64_t)(max_len + 1) * Q * 2 * h);
  off = (off + 31) & ~int64_t(31);                       // 128-byte alignment for the TMA source blocks
  w.P_row = take(umma_packed_bytes(6 * h, h) / 4);
  w.P_ent = take(umma_packed_bytes(6 * h, h) / 4);
  w.P_rel = take(umma_packed_bytes(3 * h, h) / 4);
  w.P_glob = take(umma_packed_bytes(6 * h, h) / 4);
  w.p_hh_bytes = umma_packed_bytes(3 * h, h);
  w.P_hh = take(2 * w.p_hh_bytes / 4);
  w.sync = take(32);
  w.Xd4 = w.Xd3 = w.P_x4 = w.P_x3 = w.zrow = nullptr;
  if (dropout) {
    off = (off + 31) & ~int64_t(31);
    w.P_x4 = take(umma_packed_bytes(3 * h, 4 * h) / 4);
    w.P_x3 = take(umma_packed_bytes(3 * h, 3 * h) / 4);
    w.Xd4 = take(S * 4 * h);
    w.Xd3 = take(S * 3 * h);
    w.zrow = take(S);
  }
  w.total_floats = off;
  return w;
}

constexpr int kMaxLenWs = 16;  // workspace is sized for sequences up to this long (reference: 10)

}  // namespace

int64_t gru_workspace_floats(int64_t S, int64_t Q, int64_t T, int h, bool dropout) {
  return carve(nullptr, S, Q, T, h, kMaxLenWs, dropout).total_floats;
}

int launch_gru_recur(const float* GI, const float* PQ, const float* PT, const float* bhh, const int32_t* row_glob,
                     const int32_t* seq_start, const int32_t* seq_len, const float* w_hh4, const float* w_hh3, float* Hs,
                     float* GH, float* hn4, float* hn3, unsigned int* barrier_counter, const int32_t* host_batch_sizes,
                     int max_len, int64_t Q, int h, cudaStream_t stream);

int launch_dropout_mask(uint64_t seed, uint64_t offset, int64_t n, float p, float* out, cudaStream_t stream) {
  dropout_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(seed, offset, n, p, out);
  RENET_CHECK_LAUNCH("dropout_mask_kernel");
  return RENET_OK;
}

int launch_pack_inputs(const float* H2, const int32_t* readout, const int32_t* row_glob, const float* glob,
                       const float* ent, const float* rel, const int32_t* row_seq, const int32_t* seq_s,
                       const int32_t* seq_r, const int32_t* packed_row, float* X4, float* X3, int64_t S, int h,
                       cudaStream_t stream) {
  if (S == 0) return RENET_OK;
  pack_inputs_kernel<<<(unsigned)S, 64, 0, stream>>>(H2, readout, row_glob, glob, ent, rel, row_seq, seq_s,
                                                     seq_r, packed_row, X4, X3, S, h);
  RENET_CHECK_LAUNCH("pack_inputs_kernel");
  return RENET_OK;
}

int launch_gru_fwd(const float* H2, const int32_t* readout, const int32_t* row_glob, const float* glob,
                   const float* ent, const float* rel, const int32_t* seq_s, const int32_t* seq_r,
                   const int32_t* seq_len, const int32_t* seq_start, const int32_t* host_batch_sizes,
                   int max_len, const float* w_ih4, const float* w_hh4, const float* b_ih4, const float* b_hh4,
                   const float* w_ih3, const float* w_hh3, const float* b_ih3, const float* b_hh3, float* hn4,
                   float* hn3, int64_t S, int64_t Q, int64_t T, int h, float* ws_base, cudaStream_t stream, float p_drop,
                   uint64_t seed, const int32_t* row_seq, const float* ext_X4, int k4, const float* ext_X3, int k3, int phase) {
  // phase 0: everything.  phase 1: only what does not depend on H2 (weight packing, bias rows, the per-sequence and
  // per-timestamp projections PQ / PT); phase 2: the rest (GI and the recurrence).  renet_encode_fwd runs phase 1 on a side
  // stream under the RGCN layers.  The split exists for the tensor-core engine without dropout; other configurations do
  // everything in phase 2.
  // ext_X4 != nullptr: "dense" mode -- GRU(s) on caller-materialised inputs X4 [S,k4] (and X3 [S,k3], or nullptr for a single
  // GRU: the global model's GRU(h,h), global_model.py:25,49); readout / ent / rel / glob / row_glob are not used
  const bool dense = ext_X4 != nullptr;
  if (!dense) { k4 = 4 * h; k3 = 3 * h; }
  if (max_len > kMaxLenWs) {
    set_error("renet_gru_fwd: max_len %d exceeds the supported %d", max_len, kMaxLenWs);
    return RENET_ERR_INVALID_ARG;
  }
  const bool dropout = p_drop > 0.f || dense;
  GruWs w = carve(ws_base, S, Q, T, h, kMaxLenWs, dropout);
  {
    const bool splittable = gemm_mode() != 0 && h % 4 == 0 && (3 * h) % 200 == 0 && (reinterpret_cast<uintptr_t>(ws_base) & 127) == 0 &&
                            !dropout;
    if (!splittable) {
      if (phase == 1) return RENET_OK;
      phase = 0;
    }
  }
  if (dense) {
    if (k4 <= 0 || k4 > 4 * h || k4 % 4 != 0 || (ext_X3 != nullptr && (k3 <= 0 || k3 > 3 * h || k3 % 4 != 0))) {
      set_error("renet_gru_dense_fwd: input widths must be multiples of 4 with k4 <= 4h, k3 <= 3h");
      return RENET_ERR_INVALID_ARG;
    }
    RENET_CHECK_CUDA(cudaMemsetAsync(w.zrow, 0, S * sizeof(int32_t), stream));
    row_glob = reinterpret_cast<const int32_t*>(w.zrow);          // every row reads PT row 0 (= 0)
    if (ext_X3 == nullptr) { w_ih3 = w_ih4; w_hh3 = w_hh4; b_ih3 = b_ih4; b_hh3 = b_hh4; }   // second encoder: idle copy
  }
  const dim3 tb(32, 8);
  auto pack = [&](const float* src, int ld_src, int src_off, float* dst, int ld_dst, int dst_off) -> int {
    dim3 grid((3 * h + 31) / 32, (h + 31) / 32);
    pack_transpose_kernel<<<grid, tb, 0, stream>>>(src, ld_src, src_off, 3 * h, dst, ld_dst, dst_off, h);
    RENET_CHECK_LAUNCH("pack_transpose_kernel");
    return RENET_OK;
  };
  int rc;
  // Tensor-core engine: weights go straight into the UMMA operand image (hi/lo planes, K-major, 128-byte swizzle),
  // ONCE per call -- the recurrent weights are re-used by every time step -- and every GEMM is one launch; the two
  // encoders' recurrent GEMMs are batched into a single launch per step.
  const bool use_umma = gemm_mode() != 0 && h % 4 == 0 && (3 * h) % 200 == 0 &&
                        (reinterpret_cast<uintptr_t>(ws_base) & 127) == 0;
  if (use_umma) {
    const int t3 = 3 * h / 200;   // column tiles per encoder
    // the packed images only change with the weights: with a declared weight generation they are cached across calls
    if (dense) {
      if ((rc = umma_pack_b(w_hh4, 1, h, 3 * h, h, w.P_hh, 0, stream))) return rc;
      if ((rc = umma_pack_b(w_hh3, 1, h, 3 * h, h, reinterpret_cast<uint8_t*>(w.P_hh) + w.p_hh_bytes, 0, stream))) return rc;
    } else {
      const void* keys[5] = {w_ih4, w_ih3, w_hh4, w_hh3, reinterpret_cast<const void*>((intptr_t)h)};
      const int64_t p_bytes = ((w.P_hh - w.P_row) * 4) + 2 * w.p_hh_bytes;
      bool hit = false;
      float* cached = static_cast<float*>(packed_cache_lookup(keys, 5, p_bytes, &hit));
      if (cached) {
        const float* base = w.P_row;
        w.P_ent = cached + (w.P_ent - base); w.P_rel = cached + (w.P_rel - base); w.P_glob = cached + (w.P_glob - base);
        w.P_hh = cached + (w.P_hh - base); w.P_row = cached;
      }
      if (!hit && phase != 2) {
        // logical B[k][n] = w[n][col_off + k]  ->  sk = 1, sn = leading dimension of w
        if ((rc = umma_pack_b(w_ih4, 1, 4 * h, 3 * h, h, w.P_row, 0, stream))) return rc;
        if ((rc = umma_pack_b(w_ih3, 1, 3 * h, 3 * h, h, w.P_row, t3, stream))) return rc;
        if ((rc = umma_pack_b(w_ih4 + h, 1, 4 * h, 3 * h, h, w.P_ent, 0, stream))) return rc;
        if ((rc = umma_pack_b(w_ih3 + h, 1, 3 * h, 3 * h, h, w.P_ent, t3, stream))) return rc;
        if ((rc = umma_pack_b(w_ih4 + 2 * h, 1, 4 * h, 3 * h, h, w.P_rel, 0, stream))) return rc;
        if ((rc = umma_pack_b(w_ih4 + 3 * h, 1, 4 * h, 3 * h, h, w.P_glob, 0, stream))) return rc;
        if ((rc = umma_pack_b(w_ih3 + 2 * h, 1, 3 * h, 3 * h, h, w.P_glob, t3, stream))) return rc;
        if ((rc = umma_pack_b(w_hh4, 1, h, 3 * h, h, w.P_hh, 0, stream))) return rc;
        if ((rc = umma_pack_b(w_hh3, 1, h, 3 * h, h, reinterpret_cast<uint8_t*>(w.P_hh) + w.p_hh_bytes, 0, stream))) return rc;
      }
    }
    if (phase != 2) {
      concat_bias_kernel<<<(6 * h + 255) / 256, 256, 0, stream>>>(b_ih4, b_ih3, w.bih, 3 * h);
      RENET_CHECK_LAUNCH("concat_bias_kernel");
      concat_bias_kernel<<<(6 * h + 255) / 256, 256, 0, stream>>>(b_hh4, b_hh3, w.bhh, 3 * h);
      RENET_CHECK_LAUNCH("concat_bias_kernel");
    }
    if (dropout) {
      // masked (or caller-provided) inputs materialised once, projected by two GEMMs:
      // GI = [X4 @ W_ih4^T | X3 @ W_ih3^T]; PQ = b_ih, PT = 0
      const float* X4 = dense ? ext_X4 : w.Xd4;
      const float* X3 = dense ? ext_X3 : w.Xd3;
      if ((rc = umma_pack_b(w_ih4, 1, k4, 3 * h, k4, w.P_x4, 0, stream))) return rc;
      if (X3 != nullptr && (rc = umma_pack_b(w_ih3, 1, k3, 3 * h, k3, w.P_x3, 0, stream))) return rc;
      if (!dense) {
        pack_inputs_dropout_kernel<<<(unsigned)S, 128, 0, stream>>>(H2, readout, row_glob, glob, ent, rel, row_seq, seq_s, seq_r,
                                                                   w.Xd4, w.Xd3, S, h, p_drop, seed);
        RENET_CHECK_LAUNCH("pack_inputs_dropout_kernel");
      }
      if ((rc = umma_gemm_prepacked(X4, nullptr, k4, w.P_x4, w.GI, 6 * h, nullptr, S, 3 * h, k4, false, 1, 0, 0, 0, stream))) return rc;
      if (X3 != nullptr) {
        if ((rc = umma_gemm_prepacked(X3, nullptr, k3, w.P_x3, w.GI + 3 * h, 6 * h, nullptr, S, 3 * h, k3, false, 1, 0, 0, 0, stream))) return rc;
      } else {
        RENET_CHECK_CUDA(cudaMemset2DAsync(w.GI + 3 * h, 6 * h * sizeof(float), 0, 3 * h * sizeof(float), S, stream));
      }
      fill_rows_kernel<<<(unsigned)((Q * 6 * h + 255) / 256), 256, 0, stream>>>(w.bih, w.PQ, Q, 6 * h);
      RENET_CHECK_LAUNCH("fill_rows_kernel");
      RENET_CHECK_CUDA(cudaMemsetAsync(w.PT, 0, T * 6 * h * sizeof(float), stream));
    } else {
    if (phase != 1)
      if ((rc = umma_gemm_prepacked(H2, readout, h, w.P_row, w.GI, 6 * h, nullptr, S, 6 * h, h, false, 1, 0, 0, 0, stream))) return rc;
    if (phase != 2) {
      if ((rc = umma_gemm_prepacked(ent, seq_s, h, w.P_ent, w.PQ, 6 * h, w.bih, Q, 6 * h, h, false, 1, 0, 0, 0, stream))) return rc;
      if ((rc = umma_gemm_prepacked(rel, seq_r, h, w.P_rel, w.PQ, 6 * h, nullptr, Q, 3 * h, h, true, 1, 0, 0, 0, stream))) return rc;
      if ((rc = umma_gemm_prepacked(glob, nullptr, h, w.P_glob, w.PT, 6 * h, nullptr, T, 6 * h, h, false, 1, 0, 0, 0, stream))) return rc;
    }
    }
    if (phase == 1) return RENET_OK;
    // recurrence: one persistent cooperative tensor-core kernel for all time steps and both encoders (gru_recur.cu);
    // the step-by-step loop below is the fallback for shapes it does not take
    rc = launch_gru_recur(w.GI, w.PQ, w.PT, w.bhh, row_glob, seq_start, seq_len, w_hh4, w_hh3, w.Hs, w.GH, hn4, hn3,
                          reinterpret_cast<unsigned int*>(w.sync), host_batch_sizes, max_len, Q, h, stream);
    if (rc < 0) return rc;
    if (rc == 1) return RENET_OK;
    const int64_t hs_stride_u = Q * 2 * h;
    for (int t = 0; t < max_len; ++t) {
      const int n_act = host_batch_sizes[t];
      if (n_act <= 0) break;
      const float* Hprev = (t == 0) ? nullptr : w.Hs + (int64_t)t * hs_stride_u;
      float* Hnext = w.Hs + (int64_t)(t + 1) * hs_stride_u;
      float* GH = w.GH + (int64_t)t * Q * 6 * h;
      if (t > 0) {   // both encoders in one launch: batch b reads Hprev[:, b*h:(b+1)*h], writes GH[:, b*3h:(b+1)*3h]
        if ((rc = umma_gemm_prepacked(Hprev, nullptr, 2 * h, w.P_hh, GH, 6 * h, nullptr, n_act, 3 * h, h, false, 2, h,
                                      w.p_hh_bytes, 3 * h, stream)))
          return rc;
      }
      const int total = n_act * 2 * h;
      gru_gate_kernel<<<(total + 255) / 256, 256, 0, stream>>>(w.GI, w.PQ, w.PT, GH, w.bhh, row_glob, seq_start, seq_len,
                                                              Hprev, Hnext, hn4, hn3, n_act, h, t);
      RENET_CHECK_LAUNCH("gru_gate_kernel");
    }
    return RENET_OK;
  }
  if (dropout) {
    set_error("renet_gru_fwd_dropout needs the tensor-core GEMM engine (RENET_GEMM=umma) and h %% 4 == 0, 3h %% 200 == 0");
    return RENET_ERR_INVALID_ARG;
  }
  // column blocks of W_ih: encoder x4 = [row | ent | rel | glob], encoder_r x3 = [row | ent | glob]
  if ((rc = pack(w_ih4, 4 * h, 0, w.Brow, 6 * h, 0))) return rc;
  if ((rc = pack(w_ih3, 3 * h, 0, w.Brow, 6 * h, 3 * h))) return rc;
  if ((rc = pack(w_ih4, 4 * h, h, w.Bent, 6 * h, 0))) return rc;
  if ((rc = pack(w_ih3, 3 * h, h, w.Bent, 6 * h, 3 * h))) return rc;
  if ((rc = pack(w_ih4, 4 * h, 2 * h, w.Brel, 3 * h, 0))) return rc;
  if ((rc = pack(w_ih4, 4 * h, 3 * h, w.Bglob, 6 * h, 0))) return rc;
  if ((rc = pack(w_ih3, 3 * h, 2 * h, w.Bglob, 6 * h, 3 * h))) return rc;
  if ((rc = pack(w_hh4, h, 0, w.Whh, 6 * h, 0))) return rc;
  if ((rc = pack(w_hh3, h, 0, w.Whh, 6 * h, 3 * h))) return rc;
  concat_bias_kernel<<<(6 * h + 255) / 256, 256, 0, stream>>>(b_ih4, b_ih3, w.bih, 3 * h);
  RENET_CHECK_LAUNCH("concat_bias_kernel");
  concat_bias_kernel<<<(6 * h + 255) / 256, 256, 0, stream>>>(b_hh4, b_hh3, w.bhh, 3 * h);
  RENET_CHECK_LAUNCH("concat_bias_kernel");

  // input projections
  if ((rc = sgemm_nn(H2, readout, h, w.Brow, 6 * h, w.GI, 6 * h, nullptr, S, 6 * h, h, false, stream))) return rc;
  if ((rc = sgemm_nn(ent, seq_s, h, w.Bent, 6 * h, w.PQ, 6 * h, w.bih, Q, 6 * h, h, false, stream))) return rc;
  if ((rc = sgemm_nn(rel, seq_r, h, w.Brel, 3 * h, w.PQ, 6 * h, nullptr, Q, 3 * h, h, true, stream))) return rc;
  if ((rc = sgemm_nn(glob, nullptr, h, w.Bglob, 6 * h, w.PT, 6 * h, nullptr, T, 6 * h, h, false, stream))) return rc;

  // recurrence over the packed time steps
  const int64_t hs_stride = Q * 2 * h;
  for (int t = 0; t < max_len; ++t) {
    const int n_act = host_batch_sizes[t];
    if (n_act <= 0) break;
    const float* Hprev = (t == 0) ? nullptr : w.Hs + (int64_t)t * hs_stride;
    float* Hnext = w.Hs + (int64_t)(t + 1) * hs_stride;
    float* GH = w.GH + (int64_t)t * Q * 6 * h;
    if (t > 0) {
      if ((rc = sgemm_nn(Hprev, nullptr, 2 * h, w.Whh, 6 * h, GH, 6 * h, nullptr, n_act, 3 * h, h, false, stream)))
        return rc;
      if ((rc = sgemm_nn(Hprev + h, nullptr, 2 * h, w.Whh + 3 * h, 6 * h, GH + 3 * h, 6 * h, nullptr, n_act,
                         3 * h, h, false, stream)))
        return rc;
    }
    const int total = n_act * 2 * h;
    gru_gate_kernel<<<(total + 255) / 256, 256, 0, stream>>>(w.GI, w.PQ, w.PT, GH, w.bhh, row_glob, seq_start,
                                                            seq_len, Hprev, Hnext, hn4, hn3, n_act, h, t);
    RENET_CHECK_LAUNCH("gru_gate_kernel");
  }
  return RENET_OK;
}


// ------------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------------
namespace {

// One reverse time step for both encoders.  Thread = (q < n_act, encoder, unit).
//   dh   : gradient w.r.t. the state AFTER step t: from dHcur for q < n_next (sequences that continue),
//          from dhn4/dhn3 for n_next <= q < n_act (sequences whose last step is t)
//   out  : dGI[row] (3 gates), dGH[q] (3 gates), dHprev[q] = dh * z  (the W_hh part is added by a GEMM)
__global__ void gru_gate_bwd_kernel(const float* __restrict__ GI, const float* __restrict__ PQ,
                                    const float* __restrict__ PT, const float* __restrict__ GH,
                                    const float* __restrict__ bhh, const int32_t* __restrict__ row_glob,
                                    const int32_t* __restrict__ seq_start, const float* __restrict__ Hprev,
                                    const float* __restrict__ dHcur, const float* __restrict__ dhn4,
                                    const float* __restrict__ dhn3, float* __restrict__ dGI,
                                    float* __restrict__ dGH, float* __restrict__ dHprev, float* __restrict__ Hprev_zero,
                                    int Q, int n_act, int n_next, int h, int t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int per_q = 2 * h;
  if (i >= Q * per_q) return;
  const int q = i / per_q, c = i % per_q;
  const int enc = c / h, u = c % h;
  if (q >= n_act) {
    // sequence already over at step t: its rows of this step's dGH (and of the saved state feeding the batched dW_hh
    // GEMM, whose workspace rows were never written for it) must be exact zeros
    float* z = dGH + (int64_t)q * 6 * h + enc * 3 * h + u;
    z[0] = 0.f; z[h] = 0.f; z[2 * h] = 0.f;
    if (Hprev_zero != nullptr) Hprev_zero[(int64_t)q * per_q + c] = 0.f;
    return;
  }
  const int64_t row = (int64_t)seq_start[q] + t;
  const int64_t g = (int64_t)row_glob[row];
  const int base = enc * 3 * h + u;
  const float* gi = GI + row * 6 * h + base;
  const float* pq = PQ + (int64_t)q * 6 * h + base;
  const float* pt = PT + g * 6 * h + base;
  const float i_r = gi[0] + pq[0] + pt[0];
  const float i_z = gi[h] + pq[h] + pt[h];
  const float i_n = gi[2 * h] + pq[2 * h] + pt[2 * h];
  float h_r = bhh[base], h_z = bhh[base + h], h_n = bhh[base + 2 * h], hp = 0.f;
  if (Hprev != nullptr) {
    const float* gh = GH + (int64_t)q * 6 * h + base;
    h_r += gh[0]; h_z += gh[h]; h_n += gh[2 * h];
    hp = Hprev[(int64_t)q * per_q + c];
  }
  const float r = sigmoidf_(i_r + h_r);
  const float z = sigmoidf_(i_z + h_z);
  const float n = tanhf(i_n + r * h_n);
  const float dh = (q < n_next) ? dHcur[(int64_t)q * per_q + c]
                                : (enc == 0 ? dhn4 : dhn3)[(int64_t)q * h + u];
  const float dn = dh * (1.f - z);
  const float dz = dh * (hp - n);
  const float dpre_n = dn * (1.f - n * n);
  const float dpre_z = dz * z * (1.f - z);
  const float dr = dpre_n * h_n;
  const float dpre_r = dr * r * (1.f - r);
  float* o = dGI + row * 6 * h + base;
  o[0] = dpre_r; o[h] = dpre_z; o[2 * h] = dpre_n;
  float* o2 = dGH + (int64_t)q * 6 * h + base;
  o2[0] = dpre_r; o2[h] = dpre_z; o2[2 * h] = dpre_n * r;
  dHprev[(int64_t)q * per_q + c] = dh * z;
}

// out[c] += sum_{r < n} X[r*ld + c]   (grid: column blocks x row chunks; one atomic per thread)
__global__ void colsum_accum_kernel(const float* __restrict__ X, int64_t ld, int64_t n, int cols,
                                    float* __restrict__ out, int rows_per_block) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  const int64_t r1 = min(n, r0 + rows_per_block);
  float s = 0.f;
  for (int64_t r = r0; r < r1; ++r) s += X[r * ld + c];
  atomicAdd(out + c, s);
}

// dPQ[q, :] = sum over the rows of sequence q of dGI[row, :]
__global__ void seq_rowsum_kernel(const float* __restrict__ dGI, const int32_t* __restrict__ seq_start,
                                  const int32_t* __restrict__ seq_len, float* __restrict__ dPQ, int cols) {
  const int q = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const int64_t r0 = seq_start[q];
  const int len = seq_len[q];
  float s = 0.f;
  for (int t = 0; t < len; ++t) s += dGI[(r0 + t) * cols + c];
  dPQ[(int64_t)q * cols + c] = s;
}

// dst[o, dst_off + k] += src[k, src_off + o]   (inverse of pack_transpose_kernel, accumulating)
__global__ void unpack_transpose_add_kernel(const float* __restrict__ src, int ld_src, int src_off, int rows_dst,
                                            float* __restrict__ dst, int ld_dst, int dst_off, int h) {
  __shared__ float tile[32][33];
  const int o0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;
  for (int i = ty; i < 32; i += 8) {
    int k = k0 + i, o = o0 + tx;
    tile[i][tx] = (o < rows_dst && k < h) ? src[(int64_t)k * ld_src + src_off + o] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    int o = o0 + i, k = k0 + tx;
    if (o < rows_dst && k < h) dst[(int64_t)o * ld_dst + dst_off + k] += tile[tx][i];
  }
}

struct GruBwdWs {
  float *dGI, *dGH, *dPQ, *dPT, *dHa, *dHb, *dBrow, *dBent, *dBrel, *dBglob, *dWhh, *dRows, *dQ, *dbias, *P_hhT, *dX4, *dX3;
  int64_t p_hht_bytes;
  int64_t total_floats;
};

GruBwdWs carve_bwd(float* base, int64_t S, int64_t Q, int64_t T, int h, bool dropout = false) {
  GruBwdWs w;
  int64_t off = 0;
  auto take = [&](int64_t n) { float* p = base ? base + off : nullptr; off += align4(n); return p; };
  w.dGI = take(S * 6 * h);
  w.dGH = take((int64_t)kMaxLenWs * Q * 6 * h);          // every step's recurrent-gate gradients (one dW_hh GEMM over all steps)
  w.dPQ = take(Q * 6 * h);
  w.dPT = take(T * 6 * h);
  w.dHa = take(Q * 2 * h);
  w.dHb = take(Q * 2 * h);
  w.dBrow = take((int64_t)h * 6 * h);
  w.dBent = take((int64_t)h * 6 * h);
  w.dBrel = take((int64_t)h * 3 * h);
  w.dBglob = take((int64_t)h * 6 * h);
  w.dWhh = take((int64_t)h * 6 * h);
  w.dRows = take(S * h);
  w.dQ = take(Q * h);
  w.dbias = take(12 * h);
  off = (off + 31) & ~int64_t(31);                       // 128-byte alignment for the TMA source blocks
  w.p_hht_bytes = umma_packed_bytes(h, 3 * h);
  w.P_hhT = take(2 * w.p_hht_bytes / 4);
  w.dX4 = w.dX3 = nullptr;
  if (dropout) {
    w.dX4 = take(S * 4 * h);
    w.dX3 = take(S * 3 * h);
  }
  w.total_floats = off;
  return w;
}

}  // namespace

int64_t gru_bwd_workspace_floats(int64_t S, int64_t Q, int64_t T, int h, bool dropout) {
  return carve_bwd(nullptr, S, Q, T, h, dropout).total_floats;
}

int launch_scatter_add_rows(const float* src, const int32_t* index, float* dst, int64_t n_rows, int d,
                            cudaStream_t stream);

int launch_gru_bwd(const float* H2, const int32_t* readout, const int32_t* row_glob, const float* glob,
                   const float* ent, const float* rel, const int32_t* seq_s, const int32_t* seq_r,
                   const int32_t* seq_len, const int32_t* seq_start, const int32_t* host_batch_sizes, int max_len,
                   const float* w_ih4, const float* w_hh4, const float* w_ih3, const float* w_hh3,
                   const float* dhn4, const float* dhn3, float* dH2, float* d_ent, float* d_rel, float* d_glob,
                   float* dw_ih4, float* dw_hh4, float* db_ih4, float* db_hh4, float* dw_ih3, float* dw_hh3,
                   float* db_ih3, float* db_hh3, int64_t N, int64_t S, int64_t Q, int64_t T, int h,
                   const float* fwd_ws, float* bwd_ws, cudaStream_t stream, float p_drop, uint64_t seed,
                   const int32_t* row_seq, const float* ext_X4, int k4, const float* ext_X3, int k3, float* out_dX4,
                   float* out_dX3) {
  const bool dense = ext_X4 != nullptr;
  if (!dense) { k4 = 4 * h; k3 = 3 * h; }
  const bool dropout = p_drop > 0.f || dense;
  GruWs f = carve(const_cast<float*>(fwd_ws), S, Q, T, h, kMaxLenWs, dropout);
  GruBwdWs b = carve_bwd(bwd_ws, S, Q, T, h, dropout);
  if (dense) {
    row_glob = reinterpret_cast<const int32_t*>(f.zrow);
    if (ext_X3 == nullptr) { w_ih3 = w_ih4; w_hh3 = w_hh4; }
  }
  int rc;
  RENET_CHECK_CUDA(cudaMemsetAsync(b.dbias, 0, 12 * h * sizeof(float), stream));
  RENET_CHECK_CUDA(cudaMemsetAsync(b.dWhh, 0, (int64_t)h * 6 * h * sizeof(float), stream));
  RENET_CHECK_CUDA(cudaMemsetAsync(b.dPT, 0, T * 6 * h * sizeof(float), stream));
  if (dH2 != nullptr) RENET_CHECK_CUDA(cudaMemsetAsync(dH2, 0, N * h * sizeof(float), stream));
  int last = 0;
  while (last < max_len && host_batch_sizes[last] > 0) ++last;
  if (last > kMaxLenWs) {
    set_error("renet_gru_bwd: max_len %d exceeds the supported %d", last, kMaxLenWs);
    return RENET_ERR_INVALID_ARG;
  }
  const int64_t hs_stride = Q * 2 * h;
  const int64_t gh_stride = Q * 6 * h;
  // tensor-core engine: W_hh of both encoders packed ONCE as the B operand of dHprev += dGH @ W_hh (B[k][n] = w_hh[k*h + n])
  const bool use_umma = gemm_mode() != 0 && umma_shape_ok(h, 3 * h) && (reinterpret_cast<uintptr_t>(b.P_hhT) & 127) == 0;
  if (use_umma && last > 1) {
    if ((rc = umma_pack_b(w_hh4, h, 1, h, 3 * h, b.P_hhT, 0, stream))) return rc;
    if ((rc = umma_pack_b(w_hh3, h, 1, h, 3 * h, reinterpret_cast<uint8_t*>(b.P_hhT) + b.p_hht_bytes, 0, stream))) return rc;
  }
  float* dHcur = b.dHa;
  float* dHprev = b.dHb;
  for (int t = last - 1; t >= 0; --t) {
    const int n_act = host_batch_sizes[t];
    const int n_next = (t + 1 < last) ? host_batch_sizes[t + 1] : 0;
    float* Hprev = (t == 0) ? nullptr : f.Hs + (int64_t)t * hs_stride;
    const float* GH = f.GH + (int64_t)t * gh_stride;
    float* dGHt = b.dGH + (int64_t)t * gh_stride;
    const int64_t total = Q * 2 * h;
    gru_gate_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(f.GI, f.PQ, f.PT, GH, f.bhh, row_glob, seq_start,
                                                                            Hprev, dHcur, dhn4, dhn3, b.dGI, dGHt, dHprev, Hprev,
                                                                            (int)Q, n_act, n_next, h, t);
    RENET_CHECK_LAUNCH("gru_gate_bwd_kernel");
    if (t > 0) {
      // dHprev += dGH_enc @ w_hh_enc   ([n,3h] @ [3h,h]), both encoders in one launch
      if (use_umma) {
        if ((rc = umma_gemm_prepacked(dGHt, nullptr, 6 * h, b.P_hhT, dHprev, 2 * h, nullptr, n_act, h, 3 * h, true, 2, 3 * h,
                                      b.p_hht_bytes, h, stream)))
          return rc;
      } else {
        if ((rc = sgemm_nn(dGHt, nullptr, 6 * h, w_hh4, h, dHprev, 2 * h, nullptr, n_act, h, 3 * h, true, stream))) return rc;
        if ((rc = sgemm_nn(dGHt + 3 * h, nullptr, 6 * h, w_hh3, h, dHprev + h, 2 * h, nullptr, n_act, h, 3 * h, true, stream))) return rc;
      }
    }
    float* tmp = dHcur; dHcur = dHprev; dHprev = tmp;
  }
  if (last > 0) {
    // db_hh += colsum(dGH) over every step (rows of finished sequences are zeros)
    const int rpb = 256;
    const int64_t rows = (int64_t)last * Q;
    dim3 grid((6 * h + 127) / 128, (unsigned)((rows + rpb - 1) / rpb));
    colsum_accum_kernel<<<grid, 128, 0, stream>>>(b.dGH, 6 * h, rows, 6 * h, b.dbias + 6 * h, rpb);
    RENET_CHECK_LAUNCH("colsum_accum_kernel");
  }
  if (last > 1) {
    // dWhh[k, o] += sum over steps t >= 1 of Hprev_t[:, k]^T dGH_t[:, o]: ONE K-long reduction per encoder over all steps
    const int64_t K = (int64_t)(last - 1) * Q;
    if ((rc = sgemm_tn(f.Hs + hs_stride, nullptr, 2 * h, b.dGH + gh_stride, 6 * h, b.dWhh, 6 * h, h, 3 * h, K, true, stream))) return rc;
    if ((rc = sgemm_tn(f.Hs + hs_stride + h, nullptr, 2 * h, b.dGH + gh_stride + 3 * h, 6 * h, b.dWhh + 3 * h, 6 * h, h, 3 * h, K, true, stream))) return rc;
  }
  // ---- biases of the input projection: every row carries b_ih once ------------------------------------
  {
    const int rpb = 128;
    dim3 grid((6 * h + 127) / 128, (unsigned)((S + rpb - 1) / rpb));
    colsum_accum_kernel<<<grid, 128, 0, stream>>>(b.dGI, 6 * h, S, 6 * h, b.dbias, rpb);
    RENET_CHECK_LAUNCH("colsum_accum_kernel");
  }
  if (dropout) {
    // ---- input-dropout path: dW_ih = dGI^T @ Xd (the masked inputs the forward pass kept), dXd = dGI @ W_ih, then the
    //      masks are regenerated and the gradients scattered to H2 rows / ent / rel / glob -------------------------------------
    const float* X4 = dense ? ext_X4 : f.Xd4;
    const float* X3 = dense ? ext_X3 : f.Xd3;
    float* dX4 = dense ? out_dX4 : b.dX4;
    float* dX3 = dense ? out_dX3 : b.dX3;
    if ((rc = sgemm_tn(b.dGI, nullptr, 6 * h, X4, k4, dw_ih4, k4, 3 * h, k4, S, true, stream))) return rc;
    if ((rc = sgemm_nn(b.dGI, nullptr, 6 * h, w_ih4, k4, dX4, k4, nullptr, S, k4, 3 * h, false, stream))) return rc;
    if (X3 != nullptr) {
      if ((rc = sgemm_tn(b.dGI + 3 * h, nullptr, 6 * h, X3, k3, dw_ih3, k3, 3 * h, k3, S, true, stream))) return rc;
      if ((rc = sgemm_nn(b.dGI + 3 * h, nullptr, 6 * h, w_ih3, k3, dX3, k3, nullptr, S, k3, 3 * h, false, stream))) return rc;
    }
    if (!dense) {
      unpack_inputs_dropout_kernel<<<(unsigned)S, 128, 0, stream>>>(b.dX4, b.dX3, readout, row_glob, row_seq, seq_s, seq_r, dH2,
                                                                   d_ent, d_rel, d_glob, S, h, p_drop, seed);
      RENET_CHECK_LAUNCH("unpack_inputs_dropout_kernel");
    }
    const dim3 tbd(32, 8);
    auto unpack_hh = [&](const float* src, int src_off, float* dst) -> int {
      dim3 grid((3 * h + 31) / 32, (h + 31) / 32);
      unpack_transpose_add_kernel<<<grid, tbd, 0, stream>>>(src, 6 * h, src_off, 3 * h, dst, h, 0, h);
      RENET_CHECK_LAUNCH("unpack_transpose_add_kernel");
      return RENET_OK;
    };
    if ((rc = unpack_hh(b.dWhh, 0, dw_hh4))) return rc;
    if (dw_hh3 != nullptr && (rc = unpack_hh(b.dWhh, 3 * h, dw_hh3))) return rc;
    float* outs[4] = {db_ih4, db_ih3, db_hh4, db_hh3};
    for (int k = 0; k < 4; ++k) {
      if (outs[k] == nullptr) continue;                     // single GRU: the idle second encoder has no gradients
      dim3 grid((3 * h + 127) / 128, 1);
      colsum_accum_kernel<<<grid, 128, 0, stream>>>(b.dbias + (int64_t)k * 3 * h, 3 * h, 1, 3 * h, outs[k], 1);
      RENET_CHECK_LAUNCH("colsum_accum_kernel");
    }
    return RENET_OK;
  }
  // ---- per-sequence and per-timestamp sums of dGI --------------------------------------------------------
  {
    dim3 grid((6 * h + 127) / 128, (unsigned)Q);
    seq_rowsum_kernel<<<grid, 128, 0, stream>>>(b.dGI, seq_start, seq_len, b.dPQ, 6 * h);
    RENET_CHECK_LAUNCH("seq_rowsum_kernel");
  }
  if ((rc = launch_scatter_add_rows(b.dGI, row_glob, b.dPT, S, 6 * h, stream))) return rc;
  // ---- packed weight gradients: dB = X^T @ dG ----------------------------------------------------------------
  if ((rc = sgemm_tn(H2, readout, h, b.dGI, 6 * h, b.dBrow, 6 * h, h, 6 * h, S, false, stream))) return rc;
  if ((rc = sgemm_tn(ent, seq_s, h, b.dPQ, 6 * h, b.dBent, 6 * h, h, 6 * h, Q, false, stream))) return rc;
  if ((rc = sgemm_tn(rel, seq_r, h, b.dPQ, 6 * h, b.dBrel, 3 * h, h, 3 * h, Q, false, stream))) return rc;
  if ((rc = sgemm_tn(glob, nullptr, h, b.dPT, 6 * h, b.dBglob, 6 * h, h, 6 * h, T, false, stream))) return rc;
  const dim3 tb(32, 8);
  auto unpack = [&](const float* src, int ld_src, int src_off, float* dst, int ld_dst, int dst_off) -> int {
    dim3 grid((3 * h + 31) / 32, (h + 31) / 32);
    unpack_transpose_add_kernel<<<grid, tb, 0, stream>>>(src, ld_src, src_off, 3 * h, dst, ld_dst, dst_off, h);
    RENET_CHECK_LAUNCH("unpack_transpose_add_kernel");
    return RENET_OK;
  };
  if ((rc = unpack(b.dBrow, 6 * h, 0, dw_ih4, 4 * h, 0))) return rc;
  if ((rc = unpack(b.dBrow, 6 * h, 3 * h, dw_ih3, 3 * h, 0))) return rc;
  if ((rc = unpack(b.dBent, 6 * h, 0, dw_ih4, 4 * h, h))) return rc;
  if ((rc = unpack(b.dBent, 6 * h, 3 * h, dw_ih3, 3 * h, h))) return rc;
  if ((rc = unpack(b.dBrel, 3 * h, 0, dw_ih4, 4 * h, 2 * h))) return rc;
  if ((rc = unpack(b.dBglob, 6 * h, 0, dw_ih4, 4 * h, 3 * h))) return rc;
  if ((rc = unpack(b.dBglob, 6 * h, 3 * h, dw_ih3, 3 * h, 2 * h))) return rc;
  if ((rc = unpack(b.dWhh, 6 * h, 0, dw_hh4, h, 0))) return rc;
  if ((rc = unpack(b.dWhh, 6 * h, 3 * h, dw_hh3, h, 0))) return rc;
  // biases: dbias = [db_ih4 | db_ih3 | db_hh4 | db_hh3]
  {
    float* outs[4] = {db_ih4, db_ih3, db_hh4, db_hh3};
    for (int k = 0; k < 4; ++k) {
      const int rpb = 1;
      dim3 grid((3 * h + 127) / 128, 1);
      colsum_accum_kernel<<<grid, 128, 0, stream>>>(b.dbias + (int64_t)k * 3 * h, 3 * h, 1, 3 * h, outs[k], rpb);
      RENET_CHECK_LAUNCH("colsum_accum_kernel");
    }
  }
  // ---- input gradients: dX = dG @ W_ih[:, block] ------------------------------------------------------------------
  // read-out rows -> dH2
  if ((rc = sgemm_nn(b.dGI, nullptr, 6 * h, w_ih4, 4 * h, b.dRows, h, nullptr, S, h, 3 * h, false, stream))) return rc;
  if ((rc = sgemm_nn(b.dGI + 3 * h, nullptr, 6 * h, w_ih3, 3 * h, b.dRows, h, nullptr, S, h, 3 * h, true, stream))) return rc;
  if ((rc = launch_scatter_add_rows(b.dRows, readout, dH2, S, h, stream))) return rc;
  // ent[s_q]
  if ((rc = sgemm_nn(b.dPQ, nullptr, 6 * h, w_ih4 + h, 4 * h, b.dQ, h, nullptr, Q, h, 3 * h, false, stream))) return rc;
  if ((rc = sgemm_nn(b.dPQ + 3 * h, nullptr, 6 * h, w_ih3 + h, 3 * h, b.dQ, h, nullptr, Q, h, 3 * h, true, stream))) return rc;
  if ((rc = launch_scatter_add_rows(b.dQ, seq_s, d_ent, Q, h, stream))) return rc;
  // rel[r_q]
  if ((rc = sgemm_nn(b.dPQ, nullptr, 6 * h, w_ih4 + 2 * h, 4 * h, b.dQ, h, nullptr, Q, h, 3 * h, false, stream))) return rc;
  if ((rc = launch_scatter_add_rows(b.dQ, seq_r, d_rel, Q, h, stream))) return rc;
  // glob[t]
  if (d_glob != nullptr) {
    if ((rc = sgemm_nn(b.dPT, nullptr, 6 * h, w_ih4 + 3 * h, 4 * h, d_glob, h, nullptr, T, h, 3 * h, true, stream))) return rc;
    if ((rc = sgemm_nn(b.dPT + 3 * h, nullptr, 6 * h, w_ih3 + 2 * h, 3 * h, d_glob, h, nullptr, T, h, 3 * h, true, stream))) return rc;
  }
  return RENET_OK;
}

}  // namespace renet
