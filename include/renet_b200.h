/*
 * renet_b200.h -- C-ABI of librenet_b200.so: the B200 (sm_100a) kernels behind RE-Net's
 * RGCN-aggregate + GRU hot path.
 *
 * The reference (INK-USC/RE-Net) is pure Python and has no FFI of its own; the entry points below
 * are what a binding for this path would bind -- one per arithmetic step the reference dispatches
 * to PyTorch/DGL library kernels (SURVEY.md section 2b, K1..K9).  Each declaration cites the
 * reference code it replaces (file:line under the reference tree).
 *
 * Conventions (all entry points):
 *   - plain pointers + sizes only; every pointer is a DEVICE pointer unless named host_*;
 *   - the caller owns every buffer; nothing is allocated, freed or retained by the library;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream);
 *     no hidden synchronisation, safe to capture in a CUDA graph, re-entrant, stateless;
 *   - fp32 features/weights, int32 indices (the reference uses int64; convert at the boundary);
 *   - return 0 on success, a negative renet_status otherwise; renet_last_error() (thread-local)
 *     describes the failure.  No exceptions, no exit().
 */
#ifndef RENET_B200_H
#define RENET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  RENET_OK = 0,
  RENET_ERR_INVALID_ARG = -1,   /* bad shape / null pointer / unsupported configuration        */
  RENET_ERR_CUDA = -2,          /* a CUDA runtime call or kernel launch failed                   */
  RENET_ERR_NO_DEVICE = -3      /* no sm_100 device visible                                      */
} renet_status;

/* Library version (major*10000 + minor*100 + patch). */
int renet_version(void);
/* Message for the last non-zero status returned on this thread ("" if none). */
const char* renet_last_error(void);
/* Number of kernels this library has launched on this process so far (for bench.py's
 * "gpu_launches" claim). */
int64_t renet_launch_count(void);

/* Dense-GEMM engine used for the self-loop and GRU projections: 0 = FFMA (fp32 CUDA cores),
 * 1 = tcgen05 3xTF32 (tensor cores, fp32-accurate split; the self-loop shape N = K = 200 runs a persistent kernel),
 * 2 = tcgen05 3xTF32 with the general packed kernel for every shape (the self-loop kernel before the persistent one;
 * same results, kept for A/B timing).  All are this library's own kernels.
 * Process-wide; the initial value comes from the RENET_GEMM environment variable (ffma|umma).
 * renet_set_gemm_engine returns the previous engine. */
int renet_set_gemm_engine(int engine);
int renet_get_gemm_engine(void);
/* Packed-weight cache of the tcgen05 GEMM engine.  The engine consumes weights (self-loop matrices, GRU W_ih / W_hh)
 * in a packed shared-memory operand image; packing is a kernel launch per weight per call.  Declaring a weight
 * generation >= 0 promises that every weight passed by pointer is unchanged while the generation is unchanged: packed
 * images are then kept per (device, pointers, shape) and reused, and any change of the generation invalidates all of
 * them.  generation < 0 (default) disables the cache: weights are packed on every call.  The Python host derives the
 * generation from the parameters' identities and in-place version counters. */
int renet_set_weight_generation(int64_t generation);
/* Optional caller-owned DEVICE scratch buffer (128-byte aligned) the tensor-core GEMM engine uses for the packed
 * (hi/lo split, K-major, 128-byte-swizzled) copy of the B operand, so that GEMM CTAs can fetch it with TMA bulk
 * copies.  Needs ceil(N/200)*ceil(K/32)*53248 bytes per GEMM (W_loop: 373 KB; GRU input projection: 2.2 MB); without
 * it (or if it is too small) the engine stages B itself.  The buffer is shared by all GEMMs: issue them on ONE
 * stream.  Pass NULL/0 to unregister.  The library never frees it. */
int renet_set_scratch(void* device_ptr, int64_t bytes);

/* ------------------------------------------------------------------------------------------------
 * Graph preprocessing.  Replaces what DGL does inside g.update_all (RGCN.py:91) to find the
 * in-edges of every node: turns the COO edge list of the batched history graph (dgl.batch,
 * utils.py:238) into CSR by destination.  Stable: edges of one destination keep their COO order.
 *   dst/src/etype [E] -> row_ptr [N+1], col_src [E], col_type [E], perm [E] (CSR slot -> COO edge,
 *   may be NULL).  workspace: at least renet_csr_workspace_bytes(N, E) bytes.
 * ---------------------------------------------------------------------------------------------- */
int64_t renet_csr_workspace_bytes(int64_t N, int64_t E);
int renet_build_csr(const int32_t* dst, const int32_t* src, const int32_t* etype,
                    int64_t N, int64_t E,
                    int32_t* row_ptr, int32_t* col_src, int32_t* col_type, int32_t* perm,
                    void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * RGCN block-diagonal layer, forward.
 * Replaces RGCNLayer.forward + RGCNBlockLayer.{msg_func,propagate,apply_func}
 * (RGCN.py:33-51, 79-94) and, through h_index, the embedding lookup ndata['h'] = ent_embeds[id]
 * (utils.py:239):
 *
 *   Hout[v] = act( norm[v] * sum_{e: dst(e)=v} blockdiag(W[col_type[e]]) . Hin[col_src[e]]
 *                  + Hin[v] @ Wloop )              with  Hin[v] = H[h_index ? h_index[v] : v]
 *
 *   H        [*, d_in]  row-major fp32 (rows addressed through h_index when given)
 *   h_index  [N] or NULL
 *   W        [R2, num_bases*(d_in/num_bases)*(d_out/num_bases)]  (RGCN.py:75-77 layout:
 *            block b, input i, output j at  b*si*so + i*so + j)
 *   Wloop    [d_in, d_out] or NULL (self_loop=False)
 *   row_ptr/col_src/col_type : CSR by destination (renet_build_csr); col_type already holds the
 *            column the reference selects with `reverse` (type_o if reverse else type_s,
 *            RGCN.py:80-85)
 *   norm     [N]   (1/in-degree of the batched sub-graphs, utils.py:126-127)
 *   Hout     [N, d_out]
 *   relu     1 = F.relu (layer 1), 0 = identity (layer 2)  (Aggregator.py:119-122)
 * E == 0 follows DGL 0.4: the reduce is skipped and only the apply UDF runs (agg = Hin; needs
 * d_in == d_out).  Dropout is not applied here (p = 0 / eval; see DESIGN.md).
 * ---------------------------------------------------------------------------------------------- */
int renet_rgcn_block_fwd(const float* H, const int32_t* h_index,
                         const float* W, const float* Wloop,
                         const int32_t* row_ptr, const int32_t* col_src, const int32_t* col_type,
                         const float* norm, float* Hout,
                         int64_t N, int64_t E, int32_t d_in, int32_t d_out,
                         int32_t num_bases, int32_t R2, int32_t relu, void* stream);

/* The two halves of the layer, exposed separately for profiling / tests:
 *   renet_selfloop_gemm : Hout = Hin @ Wloop                       (RGCN.py:35)
 *   renet_rgcn_gather   : Hout = act(norm * agg + (has_loop ? Hout : 0))   (RGCN.py:79-94, 45-48) */
int renet_selfloop_gemm(const float* H, const int32_t* h_index, const float* Wloop, float* Hout,
                        int64_t N, int32_t d_in, int32_t d_out, void* stream);
int renet_rgcn_gather(const float* H, const int32_t* h_index, const float* W,
                      const int32_t* row_ptr, const int32_t* col_src, const int32_t* col_type,
                      const float* norm, float* Hout,
                      int64_t N, int64_t E, int32_t d_in, int32_t d_out,
                      int32_t num_bases, int32_t R2, int32_t relu, int32_t has_loop, void* stream);
/* Same, with the caller's list of the most frequent relation ids (device int32 [n_hot], every id < R2, most frequent
 * first): at batch scale the kernel keeps the block table rows of the first few dozen of them in shared memory instead of
 * fetching a 1600-byte row per edge.  Relation frequencies are a property of the dataset (count edata['type_s'] /
 * ['type_o'] over graph_dict once); without a list (n_hot = 0, or renet_rgcn_gather) every CTA ranks the relations of its
 * own edges in its prologue.  The list only changes where a row is read from: results are bit-identical. */
int renet_rgcn_gather_hot(const float* H, const int32_t* h_index, const float* W,
                          const int32_t* row_ptr, const int32_t* col_src, const int32_t* col_type,
                          const float* norm, float* Hout,
                          int64_t N, int64_t E, int32_t d_in, int32_t d_out,
                          int32_t num_bases, int32_t R2, int32_t relu, int32_t has_loop,
                          const int32_t* hot_rel, int32_t n_hot, void* stream);
/* DEBUG ONLY (tools/stream_timeline.py): while `buffer` (device, 148 x 16 x 8 int64) is non-NULL, every batch-scale forward
 * gather launch writes per-warp time stamps into it (SM clock at entry / after the partition / first edge / last edge /
 * exit, global timer at entry and exit, edge count).  Pass NULL to switch it off; never set in production code. */
int renet_debug_stream_timing(void* buffer);

/* ------------------------------------------------------------------------------------------------
 * RGCN block-diagonal layer, backward (autograd of the above; the reference relies on
 * torch.autograd through bmm / index_select / DGL's reduce, train.py:139).
 *
 *   G = dHout * (relu ? Hout > 0 : 1)
 *   dHin[u]  += sum_{e: src(e)=u} blockdiag(W[type_e])^T . (norm[dst_e] * G[dst_e])  +  G[u] @ Wloop^T
 *   dW[r]    += sum_{e: type_e=r} Hin[src_e] (x) (norm[dst_e] * G[dst_e])     (per 2x2 block)
 *   dWloop   += Hin^T @ G
 *
 *   t_row_ptr/t_col_dst/t_col_type : CSR by SOURCE (renet_build_csr with src/dst swapped)
 *   rel_ptr [R2+1], rel_src/rel_dst [E] : edges grouped by type (renet_build_csr keyed on etype)
 *   dH       [N, d_in]   written (not accumulated); when h_index is given the caller scatters it
 *            into d(ent_embeds) with renet_scatter_add_rows
 *   dW       [R2, ...]   ACCUMULATED (+=)  -- both layers / both directions add into .grad
 *   dWloop   [d_in,d_out] ACCUMULATED (+=)
 *   G_ws     workspace of N*d_out (rounded up to a multiple of 4) + d_in*d_out floats; on return its
 *            first N*d_out floats hold P = dHout * act'(Hout)
 * ---------------------------------------------------------------------------------------------- */
int renet_rgcn_block_bwd(const float* H, const int32_t* h_index,
                         const float* W, const float* Wloop,
                         const int32_t* t_row_ptr, const int32_t* t_col_dst, const int32_t* t_col_type,
                         const int32_t* rel_ptr, const int32_t* rel_src, const int32_t* rel_dst,
                         const float* norm, const float* Hout, const float* dHout,
                         float* dH, float* dW, float* dWloop, float* G_ws,
                         int64_t N, int64_t E, int32_t d_in, int32_t d_out,
                         int32_t num_bases, int32_t R2, int32_t relu, void* stream);

/* The same backward for a graph whose destinations are a compacted subset of its nodes (the read-out sub-graph of
 * renet_readout_subgraph): H / dH have N_src rows (sources keep full-graph ids: t_row_ptr [N_src+1] is the CSR by source),
 * Hout / dHout / norm have N_dst rows (t_col_dst and rel_dst hold compact destination ids).  No self-loop part (the
 * caller runs renet_selfloop_gemm_bwd over the destination rows).  G_ws: N_dst*d_out (rounded up to 4) floats; on return
 * it holds P = dHout * act'(Hout). */
int renet_rgcn_bipartite_bwd(const float* H, const float* W,
                             const int32_t* t_row_ptr, const int32_t* t_col_dst, const int32_t* t_col_type,
                             const int32_t* rel_ptr, const int32_t* rel_src, const int32_t* rel_dst,
                             const float* norm, const float* Hout, const float* dHout,
                             float* dH, float* dW, float* G_ws,
                             int64_t N_src, int64_t N_dst, int64_t E, int32_t d_in, int32_t d_out,
                             int32_t num_bases, int32_t R2, int32_t relu, void* stream);

/* Backward of renet_selfloop_gemm:  dH = dLoop @ Wloop^T  (written),  dWloop += Hin^T @ dLoop.
 * ws: d_in*d_out floats. */
int renet_selfloop_gemm_bwd(const float* H, const int32_t* h_index, const float* Wloop,
                            const float* dLoop, float* dH, float* dWloop, float* ws,
                            int64_t N, int32_t d_in, int32_t d_out, void* stream);

/* dst[index[i], :] += src[i, :]   (gradient of the embedding lookup utils.py:239, and of the
 * read-out gather Aggregator.py:140).  d % 4 == 0. */
int renet_scatter_add_rows(const float* src, const int32_t* index, float* dst,
                           int64_t n_rows, int32_t d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Read-out + concat + GRU, forward.  Replaces Aggregator.py:139-165 (gather of the read-out rows,
 * the "# Slow!!!" concat loop, zero padding, pack_padded_sequence) and nn.GRU `encoder` /
 * `encoder_r` (model.py:28-29, 86, 94) -- only the final hidden state is produced because the
 * reference discards the per-step outputs (`tt`, model.py:86,94).
 *
 *   x4(row) = [ H2[readout[row]] | ent[seq_s[q]] | rel[seq_r[q]] | glob[row_glob[row]] ]  (4h)
 *   x3(row) = [ H2[readout[row]] | ent[seq_s[q]] |                  glob[row_glob[row]] ]  (3h)
 *   encoder  : GRU(4h -> h) over x4,  encoder_r : GRU(3h -> h) over x3, h0 = 0, gate order r,z,n.
 *
 *   Sequences are sorted by length, descending (model.py:80-81); sequence q owns rows
 *   seq_start[q] .. seq_start[q]+seq_len[q]-1 (sequence-major).  The input projection is split
 *   column-wise so the ent/rel/glob parts are computed once per sequence / per timestamp.
 *
 *   H2 [N,h]; readout [S]; row_glob [S] (row -> row of glob); glob [T,h];
 *   ent [*,h], rel [*,h] (the direction's half, model.py:66,73); seq_s, seq_r [Q];
 *   seq_len, seq_start [Q] (device, int32);  host_batch_sizes [max_len] (HOST: number of
 *   sequences active at step t -- what pack_padded_sequence computes, Aggregator.py:160-165);
 *   w_ih4 [3h,4h], w_hh4 [3h,h], b_ih4, b_hh4 [3h] : encoder;  *_3 : encoder_r ([3h,3h] ...)
 *   hn4, hn3 [Q,h] out.   workspace: renet_gru_workspace_bytes(S, Q, T, h) bytes; its contents
 *   after the call are what renet_gru_bwd needs (saved activations).
 * ---------------------------------------------------------------------------------------------- */
int64_t renet_gru_workspace_bytes(int64_t S, int64_t Q, int64_t T, int32_t h);
int renet_gru_fwd(const float* H2, const int32_t* readout, const int32_t* row_glob, const float* glob,
                  const float* ent, const float* rel, const int32_t* seq_s, const int32_t* seq_r,
                  const int32_t* seq_len, const int32_t* seq_start,
                  const int32_t* host_batch_sizes, int32_t max_len,
                  const float* w_ih4, const float* w_hh4, const float* b_ih4, const float* b_hh4,
                  const float* w_ih3, const float* w_hh3, const float* b_ih3, const float* b_hh3,
                  float* hn4, float* hn3,
                  int64_t S, int64_t Q, int64_t T, int32_t h,
                  void* workspace, int64_t workspace_bytes, void* stream);

/* Backward of renet_gru_fwd (the reference gets it from autograd through cuDNN's GRU and the concat
 * loop).  dhn4/dhn3 [Q,h]: gradients of the two final hidden states.  fwd_workspace: the workspace
 * renet_gru_fwd filled for the same inputs.  Outputs: dH2 [N,h] is WRITTEN (zero + scatter over
 * readout); d_ent [*,h], d_rel [*,h], d_glob [T,h] (may be NULL) and the eight parameter gradients
 * are ACCUMULATED (+=), like .grad. */
int64_t renet_gru_bwd_workspace_bytes(int64_t S, int64_t Q, int64_t T, int32_t h);
int renet_gru_bwd(const float* H2, const int32_t* readout, const int32_t* row_glob, const float* glob,
                  const float* ent, const float* rel, const int32_t* seq_s, const int32_t* seq_r,
                  const int32_t* seq_len, const int32_t* seq_start,
                  const int32_t* host_batch_sizes, int32_t max_len,
                  const float* w_ih4, const float* w_hh4, const float* w_ih3, const float* w_hh3,
                  const float* dhn4, const float* dhn3,
                  float* dH2, float* d_ent, float* d_rel, float* d_glob,
                  float* dw_ih4, float* dw_hh4, float* db_ih4, float* db_hh4,
                  float* dw_ih3, float* dw_hh3, float* db_ih3, float* db_hh3,
                  int64_t N, int64_t S, int64_t Q, int64_t T, int32_t h,
                  const void* fwd_workspace, void* bwd_workspace, int64_t bwd_workspace_bytes,
                  void* stream);

/* ------------------------------------------------------------------------------------------------
 * Read-out + concat + GRU with INPUT DROPOUT (training with the reference's default --dropout 0.5): Aggregator.py:157-158
 * drops elements of the two padded input tensors independently (two nn.Dropout calls on [Q,10,4h] and [Q,10,3h]) before
 * pack_padded_sequence.  With a mask per (row, column) the column-wise split of the input projection no longer applies,
 * so the masked inputs X4d [S,4h] / X3d [S,3h] are materialised once (in the workspace, kept for backward) and projected
 * by two tensor-core GEMMs; the recurrence is the same kernel as renet_gru_fwd.  Masks: Philox4x32-10 keyed by `seed`,
 * counter = element index (X4 element (row i, col c): i*4h + c; X3 element: S*4h + i*3h + c, rows sequence-major); kept
 * elements are scaled by 1/(1-p).  Nothing of the mask is stored: renet_gru_bwd_dropout regenerates it from (seed, p), and
 * renet_dropout_mask writes the same scale factors (0 or 1/(1-p)) for elements [offset, offset+n) so that tests can rebuild
 * the exact masked inputs.  The reference's own mask stream (torch's generator) cannot be reproduced; parity is exact GIVEN
 * the mask and statistical otherwise.  row_seq [S]: sequence of every row.  Needs the tensor-core GEMM engine.
 * ---------------------------------------------------------------------------------------------- */
int64_t renet_gru_dropout_workspace_bytes(int64_t S, int64_t Q, int64_t T, int32_t h);
int renet_gru_fwd_dropout(const float* H2, const int32_t* readout, const int32_t* row_glob, const float* glob,
                          const float* ent, const float* rel, const int32_t* row_seq, const int32_t* seq_s,
                          const int32_t* seq_r, const int32_t* seq_len, const int32_t* seq_start,
                          const int32_t* host_batch_sizes, int32_t max_len,
                          const float* w_ih4, const float* w_hh4, const float* b_ih4, const float* b_hh4,
                          const float* w_ih3, const float* w_hh3, const float* b_ih3, const float* b_hh3,
                          float* hn4, float* hn3, int64_t S, int64_t Q, int64_t T, int32_t h, float p, uint64_t seed,
                          void* workspace, int64_t workspace_bytes, void* stream);
int64_t renet_gru_bwd_dropout_workspace_bytes(int64_t S, int64_t Q, int64_t T, int32_t h);
int renet_gru_bwd_dropout(const float* H2, const int32_t* readout, const int32_t* row_glob, const float* glob,
                          const float* ent, const float* rel, const int32_t* row_seq, const int32_t* seq_s,
                          const int32_t* seq_r, const int32_t* seq_len, const int32_t* seq_start,
                          const int32_t* host_batch_sizes, int32_t max_len,
                          const float* w_ih4, const float* w_hh4, const float* w_ih3, const float* w_hh3,
                          const float* dhn4, const float* dhn3,
                          float* dH2, float* d_ent, float* d_rel, float* d_glob,
                          float* dw_ih4, float* dw_hh4, float* db_ih4, float* db_hh4,
                          float* dw_ih3, float* dw_hh3, float* db_ih3, float* db_hh3,
                          int64_t N, int64_t S, int64_t Q, int64_t T, int32_t h, float p, uint64_t seed,
                          const void* fwd_workspace, void* bwd_workspace, int64_t bwd_workspace_bytes, void* stream);
int renet_dropout_mask(uint64_t seed, uint64_t offset, int64_t n, float p, float* out, void* stream);

/* GRU(s) on caller-materialised inputs, final hidden states only: X4 [S,k4] for `encoder`-style weights w_ih4 [3h,k4],
 * optionally X3 [S,k3] for a second GRU run in the same launches (NULL = a single GRU: the reference's global model
 * nn.GRU(h_dim, h_dim), global_model.py:25,49; hn3 / the *_3 gradients are then scratch / NULL).  Rows are sequence-major
 * (sequence q owns rows seq_start[q] .. +seq_len[q]-1), sequences sorted by length descending, h0 = 0.  Input projection =
 * two tensor-core GEMMs, recurrence = the kernel of renet_gru_fwd.  k4 <= 4h, k3 <= 3h, multiples of 4.  Workspaces:
 * renet_gru_dropout_workspace_bytes(S, Q, 1, h) / renet_gru_bwd_dropout_workspace_bytes(S, Q, 1, h).
 * Backward: dX4 [S,k4] (dX3) written, parameter gradients accumulated. */
int renet_gru_dense_fwd(const float* X4, int32_t k4, const float* X3, int32_t k3, const int32_t* seq_len,
                        const int32_t* seq_start, const int32_t* host_batch_sizes, int32_t max_len,
                        const float* w_ih4, const float* w_hh4, const float* b_ih4, const float* b_hh4,
                        const float* w_ih3, const float* w_hh3, const float* b_ih3, const float* b_hh3,
                        float* hn4, float* hn3, int64_t S, int64_t Q, int32_t h,
                        void* workspace, int64_t workspace_bytes, void* stream);
int renet_gru_dense_bwd(const float* X4, int32_t k4, const float* X3, int32_t k3, const int32_t* seq_len,
                        const int32_t* seq_start, const int32_t* host_batch_sizes, int32_t max_len,
                        const float* w_ih4, const float* w_hh4, const float* w_ih3, const float* w_hh3,
                        const float* dhn4, const float* dhn3, float* dX4, float* dX3,
                        float* dw_ih4, float* dw_hh4, float* db_ih4, float* db_hh4,
                        float* dw_ih3, float* dw_hh3, float* db_ih3, float* db_hh3,
                        int64_t S, int64_t Q, int32_t h, const void* fwd_workspace, void* bwd_workspace,
                        int64_t bwd_workspace_bytes, void* stream);

/* Per-graph pooling over a batched graph: out[g] = max (mode 1) or mean (mode 0) of H[seg_ptr[g] .. seg_ptr[g+1]) -- dgl.max_nodes /
 * dgl.mean_nodes of the reference's global aggregator (Aggregator.py:58-61).  argmax [G,d] (mode 1) keeps the winning row for
 * backward; renet_segment_pool_bwd writes dH [N,d] (zeros elsewhere). */
int renet_segment_pool_fwd(const float* H, const int32_t* seg_ptr, int64_t G, int32_t d, int32_t mode, float* out,
                           int32_t* argmax, void* stream);
int renet_segment_pool_bwd(const float* dout, const int32_t* seg_ptr, const int32_t* argmax, int64_t G, int64_t N,
                           int32_t d, int32_t mode, float* dH, void* stream);

/* ------------------------------------------------------------------------------------------------
 * HOST-side batching of history graphs (no CUDA; every pointer here is a HOST pointer).  Replaces
 * utils.get_sorted_s_r_embed_rgcn / get_s_r_embed_rgcn minus the embedding lookups (utils.py:209-283):
 * get_neighs_by_t :149-156, get_g_list_id + make_subgraph :158-170,115-131, get_node_ids_to_g_id
 * :172-181, dgl.batch :238, and the pack_padded_sequence bookkeeping of Aggregator.py:160-165.
 *
 * Graph store (built once from graph_dict): graph g owns nodes g_node_off[g]..g_node_off[g+1]
 * (g_node_ent ascending) and edges g_edge_off[g].. (LOCAL rows g_src/g_dst, sorted by g_dst, with
 * g_type_s / g_type_o).  History store (built once from the s_hist / s_hist_t lists): sample i owns
 * the entry ids h_samp_entry[h_samp_off[i] .. h_samp_off[i+1]) (entries are shared between samples, as
 * the reference's lists share arrays); entry e happened in graph h_ent_graph[e], its subject sits at
 * local row h_ent_srow[e], its neighbours at local rows h_nbr_row[h_ent_off[e] .. h_ent_off[e+1]).
 *
 * Output: s_idx_out [B] (sample order: history length descending, stable, when sort != 0), the batched
 * graph in CSR form + bookkeeping packed into `out` (int32 words, one H2D copy):
 *   node_ent[N] row_ptr[N+1] col_src[E] col_type_s[E] col_type_o[E] norm[N](float bits)
 *   readout[S] row_comp[S] row_seq[S] seq_start[Q] seq_len[Q] packed_row[S]
 *   comp_ptr[G+1] comp_order[G] rel_slot_s[R2] hot_s[n_hot_max] rel_slot_o[R2] hot_o[n_hot_max]
 *   s_idx[B] comp_graph[G]
 * (the comp/rel line feeds renet_rgcn_gather_comp: components largest-first, and the n_hot_max most frequent
 * edge types of the batch for each type column).  comp_graph_out [G] (graph index of every component,
 * first-appearance order), batch_sizes_out [max_len],
 * sizes [10] = {N, E, S, Q, G, max_len, words_used, n_hot_s, n_hot_o, 0}.
 * Returns 0, or 1 when out_capacity < words_used (sizes is filled: grow and call again), <0 on error.
 * ---------------------------------------------------------------------------------------------- */
/* Threads renet_host_assemble_batch may use per call (default 8; use 1 when many calls run concurrently, e.g.
 * from a prefetching loader).  Returns the previous value. */
int renet_set_host_threads(int n);
int renet_host_assemble_batch(
    int64_t T, const int64_t* g_node_off, const int32_t* g_node_ent, const int64_t* g_edge_off,
    const int32_t* g_src, const int32_t* g_dst, const int32_t* g_type_s, const int32_t* g_type_o,
    const int64_t* h_samp_off, const int64_t* h_samp_entry, const int32_t* h_ent_graph, const int32_t* h_ent_srow,
    const int64_t* h_ent_off, const int32_t* h_nbr_row,
    const int64_t* sample_idx, int64_t B, int32_t sort, int32_t R2, int32_t n_hot_max,
    int64_t* s_idx_out, int32_t* out, int64_t out_capacity, int32_t* comp_graph_out,
    int32_t* batch_sizes_out, int32_t max_len_capacity, int64_t* sizes);

/* ------------------------------------------------------------------------------------------------
 * Device batcher: the same contract as renet_host_assemble_batch (reference utils.py:149-181,209-244), split so
 * that only the O(S + nodes) part runs on the host and the O(edges) part -- utils.make_subgraph's induced-edge
 * filter (utils.py:115-131) over every touched timestamp + dgl.batch (utils.py:238) -- runs on the GPU against a
 * graph store resident in HBM.
 *
 * renet_host_plan_batch (host, no CUDA): orders the samples, picks the components, marks and numbers the nodes.
 * `out` (int32 words, one H2D copy):
 *   newid[M] node_ent[N] readout[S] row_comp[S] row_seq[S] seq_start[Q] seq_len[Q] packed_row[S] s_idx[B]
 *   comp_graph[G] mark_off[G+1] cand_off[G+1]
 * newid: per component c one word per local row of its graph (at mark_off[c]): batched node id, or -1;
 * cand_off: prefix sum of the components' un-induced edge counts.  sizes [10] = {N, E_cand, S, Q, G, max_len,
 * words_used, M, 0, 0}.  Returns 0, 1 when out_capacity < words_used (grow, call again), <0 on error.
 *
 * renet_induce_edges (device pointers only): filters the E_cand candidate edges and writes the batched graph's
 * CSR by destination -- row_ptr [N+1], col_src / col_type_s / col_type_o (capacity E_cand, the first E entries
 * are valid), norm [N] = 1/max(in-degree,1) (utils.py:126-127) -- and the edge count E into e_count[0].
 * Identical, bit for bit, to renet_host_assemble_batch's output.
 * ---------------------------------------------------------------------------------------------- */
int renet_host_plan_batch(
    int64_t T, const int64_t* g_node_off, const int32_t* g_node_ent, const int64_t* g_edge_off,
    const int64_t* h_samp_off, const int64_t* h_samp_entry, const int32_t* h_ent_graph, const int32_t* h_ent_srow,
    const int64_t* h_ent_off, const int32_t* h_nbr_row, const int64_t* sample_idx, int64_t B, int32_t sort,
    int64_t* s_idx_out, int32_t* out, int64_t out_capacity, int32_t* batch_sizes_out, int32_t max_len_capacity,
    int64_t* sizes);
int64_t renet_induce_workspace_bytes(int64_t e_cand);
int renet_induce_edges(const int64_t* g_edge_off, const int32_t* g_src, const int32_t* g_dst,
                       const int32_t* g_type_s, const int32_t* g_type_o, const int32_t* comp_graph,
                       const int32_t* mark_off, const int32_t* cand_off, const int32_t* newid, int64_t G,
                       int64_t N, int64_t e_cand, int32_t* row_ptr, int32_t* col_src, int32_t* col_type_s,
                       int32_t* col_type_o, float* norm, int32_t* e_count, void* workspace,
                       int64_t workspace_bytes, void* stream);

/* Native loader: a pool of C++ worker threads that run renet_host_plan_batch / renet_host_assemble_batch jobs ahead of
 * the consumer (the reference builds every batch synchronously inside forward(), utils.py:209-244).  submit returns a
 * ticket (>= 0); every pointer passed must stay valid until renet_loader_wait returns for that ticket; wait blocks
 * until the job has run and returns the job's return code.  Jobs start in submission order. */
void* renet_loader_create(int32_t n_threads);
void renet_loader_destroy(void* loader);
int64_t renet_loader_submit_plan(
    void* loader, int64_t T, const int64_t* g_node_off, const int32_t* g_node_ent, const int64_t* g_edge_off,
    const int64_t* h_samp_off, const int64_t* h_samp_entry, const int32_t* h_ent_graph, const int32_t* h_ent_srow,
    const int64_t* h_ent_off, const int32_t* h_nbr_row, const int64_t* sample_idx, int64_t B, int32_t sort,
    int64_t* s_idx_out, int32_t* out, int64_t out_capacity, int32_t* batch_sizes_out, int32_t max_len_capacity,
    int64_t* sizes);
int64_t renet_loader_submit_assemble(
    void* loader, int64_t T, const int64_t* g_node_off, const int32_t* g_node_ent, const int64_t* g_edge_off,
    const int32_t* g_src, const int32_t* g_dst, const int32_t* g_type_s, const int32_t* g_type_o,
    const int64_t* h_samp_off, const int64_t* h_samp_entry, const int32_t* h_ent_graph, const int32_t* h_ent_srow,
    const int64_t* h_ent_off, const int32_t* h_nbr_row, const int64_t* sample_idx, int64_t B, int32_t sort, int32_t R2,
    int32_t n_hot_max, int64_t* s_idx_out, int32_t* out, int64_t out_capacity, int32_t* comp_graph_out,
    int32_t* batch_sizes_out, int32_t max_len_capacity, int64_t* sizes);
int renet_loader_wait(void* loader, int64_t ticket);

/* Sequence ids of a batch in processing order, on the device, in one launch (model.py:81-84, utils.py:224-225):
 *   seq_s[q] = triplets[s_idx[q]][col_s], seq_r[q] = triplets[s_idx[q]][1]   for q < Q   (triplets int64 [B,ld], ld >= 3;
 *   col_s = 0 for the subject direction, 2 for the object direction; s_idx = renet_host_*_batch's sample order)
 *   row_graph[i] = comp_graph[row_comp[i]]                                    for i < S   (graph-store index of the
 *   timestamp of every read-out row: indexes a dense [T_all,h] table of the global embeddings) */
int renet_prepare_sequences(const int64_t* triplets, int32_t ld, int32_t col_s, const int32_t* s_idx, int64_t Q,
                            const int32_t* comp_graph, const int32_t* row_comp, int64_t S, int32_t* seq_s,
                            int32_t* seq_r, int32_t* row_graph, void* stream);

/* One call for the whole forward hot path of one direction (inference / no autograd):
 *   H1 = relu-layer(ent[node_ent]), H2 = linear-layer(H1)   (renet_rgcn_block_fwd x2, Aggregator.py:136-137)
 *   hn4, hn3 = renet_gru_fwd(H2, ...)                          (Aggregator.py:139-165 + model.py:86,94)
 * Same arguments as the individual entry points; H1/H2 [N,h] are caller-provided outputs.  With a read-out sub-graph
 * (sub_* = the outputs of renet_readout_subgraph for this batch and type column; all NULL = none) layer 2 runs on it:
 * H2 then holds S compact rows and the GRU reads them through sub_readout.  hot_rel / n_hot: the optional relation ranking
 * of renet_rgcn_gather_hot (NULL / 0 = none), used by both layers.
 * Stream behaviour: the part of the GRU that does not depend on H2 (weight packing, bias rows, the per-sequence and
 * per-timestamp projections) is enqueued on a library-owned side stream that forks from `stream` by an event at entry and
 * joins it by an event before the H2 projection; from the caller's point of view everything is ordered on `stream`. */
int renet_encode_fwd(const float* ent, const int32_t* node_ent, const int32_t* row_ptr, const int32_t* col_src,
                     const int32_t* col_type, const float* norm,
                     const float* W1, const float* Wloop1, const float* W2, const float* Wloop2,
                     float* H1, float* H2, int64_t N, int64_t E, int32_t R2,
                     const int32_t* readout, const int32_t* row_glob, const float* glob, const float* rel,
                     const int32_t* seq_s, const int32_t* seq_r, const int32_t* seq_len, const int32_t* seq_start,
                     const int32_t* host_batch_sizes, int32_t max_len,
                     const float* w_ih4, const float* w_hh4, const float* b_ih4, const float* b_hh4,
                     const float* w_ih3, const float* w_hh3, const float* b_ih3, const float* b_hh3,
                     float* hn4, float* hn3, int64_t S, int64_t Q, int64_t T, int32_t h, int32_t num_bases,
                     const int32_t* sub_uniq, const int32_t* sub_readout, const int32_t* sub_row_ptr,
                     const int32_t* sub_col_src, const int32_t* sub_col_type, const float* sub_norm,
                     const int32_t* hot_rel, int32_t n_hot,
                     void* workspace, int64_t workspace_bytes, void* stream);

/* Materialise the packed GRU inputs exactly as the reference's aggregator returns them
 * (PackedSequence.data, time-major: Aggregator.py:160-165):  X4 [S,4h], X3 [S,3h];
 * packed_row [S] maps packed position -> sequence-major row. */
int renet_pack_inputs(const float* H2, const int32_t* readout, const int32_t* row_glob,
                      const float* glob, const float* ent, const float* rel,
                      const int32_t* row_seq, const int32_t* seq_s, const int32_t* seq_r,
                      const int32_t* packed_row, float* X4, float* X3,
                      int64_t S, int32_t h, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Read-out sub-graph.  The reference runs layer 2 of the aggregator on every node of the batched graph and then keeps the
 * read-out rows only (Aggregator.py:139-140: embeds_mean[node_ids_graph], 26 % of the rows at ICEWS18 scale).  Layer 2 at a
 * read-out node depends on layer 1 at its in-neighbours only, so layer 2 over the sub-graph {edges whose destination is a
 * read-out node} is identical on every consumed row (SURVEY.md section 8(a), optimisation (i)).  Built on the device, no
 * host round trip; launches are sized by the capacities, the actual sizes come back in counts:
 *   readout [S] -> uniq [S] (distinct read-out nodes ascending = compact destination -> node; unused tail = 0),
 *   readout_c [S] (read-out row -> compact destination), row_ptr2 [S+1] (CSR by compact destination; unused
 *   destinations have no edges), col_src2 / col_type2 (capacity of col_src; sources keep full-graph ids), norm2 [S]
 *   (tail 1), counts [2] = {U, E2}.
 * Layer 2 is then renet_selfloop_gemm(H1, uniq, ...) + renet_rgcn_gather(H1, NULL, W2, row_ptr2, col_src2, col_type2,
 * norm2, H2c, S, ...) and the GRU reads H2c through readout_c.
 * ---------------------------------------------------------------------------------------------- */
int64_t renet_readout_subgraph_workspace_bytes(int64_t N, int64_t S);
int renet_readout_subgraph(const int32_t* readout, int64_t S, int64_t N,
                           const int32_t* row_ptr, const int32_t* col_src, const int32_t* col_type, const float* norm,
                           int32_t* uniq, int32_t* readout_c, int32_t* row_ptr2, int32_t* col_src2, int32_t* col_type2,
                           float* norm2, int32_t* counts, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Decoder: logits = X @ W^T + bias followed by cross-entropy (reference model.py:89-91: object prediction, X = [ent[s] |
 * s_h | rel[r]] [B,3h], W = linear.weight [|E|,3h]; model.py:97-100: relation prediction, [B,2h] x [R,2h]).
 *   renet_decoder_ce_fwd : loss_rows[i] = logsumexp_c(logits[i,c]) - logits[i,target[i]], lse[i] = the logsumexp (kept for
 *       backward).  tcgen05 3xTF32 GEMM with a fused epilogue: the [B,|E|] logits never reach memory.
 *   renet_decoder_ce_bwd : for loss = scale * d_scale[0] * sum_i loss_rows[i] (the reference's mean: scale = 1/B; d_scale =
 *       optional DEVICE scalar, the upstream gradient, so that autograd needs no host read): dX [M,K] written; dW [N,K] and dbias [N] (may be NULL) ACCUMULATED.  The logits are recomputed; the
 *       gradient of the logits (M x N floats, row-major and transposed) lives in the workspace only.
 * K % 4 == 0; N is arbitrary (23033 classes).  X [M,K], W [N,K] row-major, 16-byte aligned; target int32 [M].
 * ---------------------------------------------------------------------------------------------- */
int64_t renet_decoder_ce_workspace_bytes(int64_t M, int32_t N, int32_t K);
int renet_decoder_ce_fwd(const float* X, const float* W, const float* bias, const int32_t* target, float* loss_rows,
                         float* lse, int64_t M, int32_t N, int32_t K, void* workspace, int64_t workspace_bytes, void* stream);
int64_t renet_decoder_ce_bwd_workspace_bytes(int64_t M, int32_t N, int32_t K);
int renet_decoder_ce_bwd(const float* X, const float* W, const float* bias, const int32_t* target, const float* lse,
                         float scale, const float* d_scale, float* dX, float* dW, float* dbias, int64_t M, int32_t N, int32_t K, void* workspace,
                         int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Optimiser step of the reference training loop on FLAT fp32 buffers (reference train.py:140-142:
 * torch.nn.utils.clip_grad_norm_(model.parameters(), grad_norm); Adam(lr, weight_decay).step()).  The data-parallel
 * engine keeps all parameters / gradients as views into one flat buffer each (the gradient buffer is what NCCL
 * all-reduces), so the step is two HBM-bound launches.
 *   renet_grad_sumsq : out[0] (=|+=) sum(grad[i]^2), fixed-order reduction (reproducible, no float atomics);
 *                      workspace: renet_grad_sumsq_workspace_bytes() bytes.
 *   renet_adam_step  : g = grad*grad_scale*clip (+ weight_decay*param);  clip = min(1, max_norm/(sqrt(sumsq[0])*grad_scale
 *                      + 1e-6)) when sumsq != NULL and max_norm > 0, else 1;  m,v moments; bias correction with `step`
 *                      (counts from 1); param updated in place.  Matches torch.optim.Adam (amsgrad=False).
 * ---------------------------------------------------------------------------------------------- */
int64_t renet_grad_sumsq_workspace_bytes(void);
int renet_grad_sumsq(const float* grad, int64_t n, float* out, int32_t accumulate, void* workspace,
                     int64_t workspace_bytes, void* stream);
int renet_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                    float beta1, float beta2, float eps, float weight_decay, int64_t step, const float* sumsq,
                    float max_norm, float grad_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RENET_B200_H */
