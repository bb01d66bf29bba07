/*
 * mlg_b200.h -- C ABI of libmlg_b200.so: hand-written sm_100a kernels for the message-passing and
 * cross-level pooling hot path of Y-Claw/Multilevel-GNN.
 *
 * The reference has no FFI / plugin table of its own (pure Python on torch_geometric /
 * torch_scatter / ATen, SURVEY.md section 8b): every entry point below replaces a chain of third-party
 * kernels reached from the cited reference call site, and is what a maintainer would bind (ctypes,
 * see INTEGRATION.md) from the reference's own nn.Module methods.
 *
 * Conventions
 *   - all pointers are DEVICE pointers on the current CUDA device unless stated otherwise;
 *     the caller allocates every output and workspace; nothing is allocated or freed inside;
 *   - float = fp32, row-major, contiguous; node/edge ids inside kernels are int32;
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work (no host sync),
 *     are re-entrant across streams/devices and safe under CUDA-graph capture
 *     (except where a function says it synchronises);
 *   - return value 0 = ok, negative = error (MLG_ERR_*); mlg_last_error() gives a thread-local text.
 */
#ifndef MLG_B200_H
#define MLG_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLG_ABI_VERSION 1

/* aggregation modes of GenMessagePassing.aggregate (models/gcn_lib/sparse/torch_message.py:44-85) */
#define MLG_AGGR_SOFTMAX 0 /* softmax, softmax_sg (learn_t=0), softmax_sum (y_dev != NULL) */
#define MLG_AGGR_POWER 1   /* power, power_sum (y_dev != NULL) */
#define MLG_AGGR_ADD 2
#define MLG_AGGR_MEAN 3
#define MLG_AGGR_MAX 4

/* epilogues of GENConv.forward (models/gcn_lib/sparse/torch_vertex.py:86-89) */
#define MLG_EPI_NONE 0     /* only the aggregated message m */
#define MLG_EPI_RESIDUAL 1 /* h = x + m */
#define MLG_EPI_MSGNORM 2  /* h = x + msg_scale * ||x||_2 * m / max(||m||_2, 1e-12) (torch_message.py:175-179) */

int mlg_abi_version(void);
const char* mlg_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * CSR construction.  Replaces per-forward remove_self_loops/add_self_loops
 * (torch_vertex.py:272-273) and the implicit index broadcast inside torch_scatter.
 *
 * edge_index: int64 [2, E] (row 0 = source j, row 1 = target i).  Builds the target-sorted CSR
 *   rowptr int32 [n_rows+1], col int32 [cap] (source of each entry), eid int32 [cap]
 *   (index of the entry's original edge, -1 for an added self loop), cap = E + (add_self ? n_rows : 0).
 * Entries of a row keep original edge order (stable), added self loops come last.
 * With by_source != 0 the roles of the two rows are swapped (CSR of the reversed graph: rows =
 * sources, col = targets) -- that is the structure the backward passes traverse.
 * drop_self removes i==j edges; the number of valid entries is rowptr[n_rows] (stays on device).
 * workspace: at least mlg_csr_build_workspace_bytes(E, n_rows, add_self) bytes.
 */
int64_t mlg_csr_build_workspace_bytes(int64_t n_edges, int64_t n_rows, int add_self);
int mlg_csr_build(const int64_t* edge_index, int64_t n_edges, int64_t n_rows, int by_source,
                  int drop_self, int add_self, int32_t* rowptr, int32_t* col, int32_t* eid,
                  void* workspace, int64_t workspace_bytes, void* stream);

/* val[q] = eid[q] >= 0 ? edge_attr[eid[q]] : fill   for q < rowptr[n_rows] (edge weights in CSR order;
 * add_self_loops fills new loops with 1.0). */
int mlg_edge_values(const float* edge_attr, const int32_t* eid, const int32_t* rowptr, int64_t n_rows,
                    int64_t cap, float fill, float* val, void* stream);

/* ---------------------------------------------------------------------------------------------
 * GENConv message + aggregation + MsgNorm/residual epilogue, forward.
 * Replaces GENConv.message (torch_vertex.py:94-101), GenMessagePassing.aggregate
 * (torch_message.py:44-85), MsgNorm.forward (torch_message.py:175-179) and `h = x + m`
 * (torch_vertex.py:89):
 *     msg_e = relu(x[col] + e[eid]) + eps            (e may be NULL)
 *     msg_e = e[eid]                                 when x == NULL: messages given directly, the
 *                                                    GenMessagePassing.aggregate(inputs, index) drop-in
 *     m_i   = AGGR_{e -> i} msg_e                    per channel, one pass, online softmax
 *     h_i   = epilogue(x_i, m_i)
 * x [n, H]; e [E, H] indexed by eid[q] (or by q when eid == NULL); t/p/y: device scalars when the
 * *_dev pointer is non-NULL (learnable Parameters), else the host value; y_dev != NULL multiplies
 * the result by deg^sigmoid(y) (softmax_sum / power_sum).
 * Outputs: m [n,H] (may be NULL for inference when h is produced); aux [n,H] (may be NULL for inference: softmax -> log2-sum-exp of t*msg*log2(e),
 * power -> the un-clamped mean); h [n,H] (NULL iff epilogue == MLG_EPI_NONE).
 */
int mlg_gen_aggr_fwd(const float* x, const float* e, const int32_t* rowptr, const int32_t* col,
                     const int32_t* eid, int64_t n, int64_t H, int mode, float t, const float* t_dev,
                     float p, const float* p_dev, const float* y_dev, float eps, int epilogue,
                     const float* msg_scale_dev, float* m, float* aux, float* h, void* stream);

/* number of float4 partial-sum rows mlg_gen_aggr_bwd writes (one per thread block) */
int64_t mlg_gen_aggr_bwd_partial_rows(int64_t n, int64_t H);

/* Backward of the above (autograd of the same reference lines; closed forms in SURVEY.md App. B).
 * g [n,H]: gradient w.r.t. h (or w.r.t. m when epilogue == MLG_EPI_NONE).
 * Writes g_edge[eid[q]] (or [q]) = d/d(pre-activation of edge q) for every entry  -- this IS the
 * gradient of e, and the rows the source-side pass (mlg_gather_sum over the by-source CSR) sums into
 * g_x; writes g_x [n,H] = the direct (residual / MsgNorm) term, zeros for MLG_EPI_NONE;
 * partials [rows,4] per block: (dL/dt or dL/dp, dL/dy_raw, dL/dmsg_scale, 0).
 * learn != 0: gradients flow through the softmax weights (learn_t) / to p (learn_p).
 */
int mlg_gen_aggr_bwd(const float* g, const float* x, const float* e, const int32_t* rowptr,
                     const int32_t* col, const int32_t* eid, int64_t n, int64_t H, int mode, int learn,
                     float t, const float* t_dev, float p, const float* p_dev, const float* y_dev,
                     float eps, int epilogue, const float* msg_scale_dev, const float* m,
                     const float* aux, float* g_edge, float* g_x, float* partials, void* stream);

/* Same backward with the source-side sum done inside the kernel (softmax family, H = 128 or 256, messages built from x:
 * mlg_gen_aggr_bwd_src_supported): g_x [n,H] = direct term + sum over out-edges of g_edge, accumulated with 16-byte
 * vector reductions into L2 (g_x is zeroed by the call) -- no second pass over g_edge [E,H].  g_edge may be NULL when the
 * caller does not need the edge gradients.  The order of the additions, hence the last bits of g_x, is not reproducible
 * (as with the reference's scatter-add backward, torch_scatter behind gcn_lib/sparse/torch_message.py:44-85). */
int mlg_gen_aggr_bwd_src_supported(int64_t H, int mode, int have_x);
int mlg_gen_aggr_bwd_src(const float* g, const float* x, const float* e, const int32_t* rowptr,
                         const int32_t* col, const int32_t* eid, int64_t n, int64_t H, int mode, int learn,
                         float t, const float* t_dev, float p, const float* p_dev, const float* y_dev,
                         float eps, int epilogue, const float* msg_scale_dev, const float* m,
                         const float* aux, float* g_edge, float* g_x, float* partials, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Weighted segment gather-sum (CSR SpMM with feature rows), all matrices row-major with a leading
 * dimension (floats) so that halves of a concatenated buffer can be read / written in place:
 *     out_i = addend_i + post_i * ( sum_{q in row i} val[q] * pre[idx[q]] * src[idx[q]] )
 *     relative != 0:  out_i -= src_i * (post_mode==mean ? 1 : cnt_i)      (RSAGE x_j*w - x_i)
 *     self_out != NULL: self_out_i = src_i                                 (left half of cat(x, agg))
 *     mask != NULL:     out_i *= (mask_i > 0 ? 1 : mask_slope) elementwise  (backward only: the derivative of the
 *                       (Leaky)ReLU that produced this layer's input, so the previous layer gets dL/dz directly)
 * val NULL = 1, pre NULL = 1, addend NULL = 0; post_mode 0: post_i = 1, 1: post_i = 1/cnt_i (cnt_i = row
 * length, PyG mean aggregation incl. the self loop), 2: post_i = post[i].
 * replicas = B > 1: the CSR (n_rows rows, idx in [0, n_rows)) is ONE graph shared by B stacked copies
 * (train.py batches: dataloader/multiloader.py:687-698); replica b gathers src rows b*rep_rows_src + idx and
 * writes out / self_out / addend rows b*n_rows + i; post is per single-graph row; pre is shared
 * (rep_rows_pre == 0) or per replica (pre[b*rep_rows_pre + idx]).  rep_rows_src == 0 is the rank-1 source
 * of MultilevelGNN's first layer: every replica reads the SAME src rows (node_embedding) scaled by its own
 * pre (batch.x), so x0 = x * node_embedding (multilevel_gnn.py:150-151) is never materialised; self_out
 * then receives pre[b*rep_rows_pre + i] * src_i.
 * order (NULL ok): int32 [n_rows] visiting order of the rows (heavy rows first; load balance only).
 * Forward use: SAGEConv mean aggregation of w_ij * x_j (torch_vertex.py:279-286 + PyG mean), done
 * BEFORE the lin_r GEMM (algebraically identical, SURVEY App. B.4).  Backward use: the same call on
 * the by-source CSR.  Also the source-side pass of mlg_gen_aggr_bwd.
 */
int mlg_gather_sum(const float* src, int64_t ld_src, const int32_t* rowptr, const int32_t* idx, const float* val,
                   const float* pre, const float* post, const int32_t* order, int64_t n_rows, int64_t C,
                   int64_t replicas, int64_t rep_rows_src, int64_t rep_rows_pre, int post_mode, int relative,
                   const float* addend, int64_t ld_add, float* out, int64_t ld_out, float* self_out,
                   int64_t ld_self, const float* mask, int64_t ld_mask, float mask_slope, const float* reduce_scale,
                   void* stream);
/* mlg_gather_sum with a fused output activation (replicated path, no relative / reduce_scale): act != 0 applies
 * out = LeakyReLU_act_slope(out) after the addend / mask steps.  Forward of a SAGE layer evaluated transform-first
 * (out_channels < in_channels: z = U + mean_j(w_ij V_j) with [U | V] = x [W1 ; W2 W_r]^T + [b | 0], so the gather runs on
 * the narrower rows). */
int mlg_gather_sum_act(const float* src, int64_t ld_src, const int32_t* rowptr, const int32_t* idx, const float* val,
                       const float* pre, const float* post, const int32_t* order, int64_t n_rows, int64_t C,
                       int64_t replicas, int64_t rep_rows_src, int64_t rep_rows_pre, int post_mode, int relative,
                       const float* addend, int64_t ld_add, float* out, int64_t ld_out, float* self_out,
                       int64_t ld_self, const float* mask, int64_t ld_mask, float mask_slope, const float* reduce_scale,
                       int act, float act_slope, void* stream);
/* reduce_scale != NULL (replicated path only): instead of one output row per (replica, row) the kernel writes, per row,
 * the weighted sum over the replicas of each replica SLICE:  out[s*n_rows + i] = sum_{b in slice s} reduce_scale[b*n_rows + i]
 * * out_i(b); out must hold mlg_gather_sum_slices(n_rows, C, replicas) * n_rows rows and the caller adds the slices.
 * This is the gradient of MultilevelGNN's embed-scale prologue (x0 = x * node_embedding, multilevel_gnn.py:150-151)
 * folded into the first layer's backward aggregation: g_emb[n,:] = sum_b x[b,n] * g_x0[b,n,:]. */
int64_t mlg_gather_sum_slices(int64_t n_rows, int64_t C, int64_t replicas);
/* The replicated aggregation over a NODE-MAJOR source of 32-wide rows: src row of (replica b, node j) is j * replicas + b (the
 * replica rows one CSR entry gathers are contiguous); out / self_out rows are graph-major (b * n_rows + i) like everywhere else.
 * out_i(b) = sum_q val_q * pre[idx_q] * src[idx_q, b];  self_out_i(b) = src[i, b] (NULL ok); val / pre / order NULL ok.
 * Backward aggregation of a transform-first SAGE layer on the gradient written by mlg_pool_bwd_layout(gx_node_major = 1). */
int mlg_gather_sum_nm(const float* src, const int32_t* rowptr, const int32_t* idx, const float* val, const float* pre,
                      const int32_t* order, int64_t n_rows, int64_t replicas, float* out, int64_t ld_out, float* self_out,
                      int64_t ld_self, void* stream);
/* The general form: src / addend node-major with leading dimensions (e.g. the V / U halves of a [rows, 64] GEMM output),
 * out_i(b) = act( addend_i(b) + post_i * sum ), post_i = 1 / row length when mean != 0, LeakyReLU(act_slope) when act != 0,
 * out / self_out node-major too when out_node_major != 0.  Forward of the transform-first SAGE layer whose input came
 * node-major from mlg_sage_rank1_fwd_rows_nm, and its backward aggregation writing [g_U | g_V] in the same row order. */
int mlg_gather_sum_nm_ex(const float* src, int64_t ld_src, const int32_t* rowptr, const int32_t* idx, const float* val,
                         const float* pre, const int32_t* order, int64_t n_rows, int64_t replicas, int mean, const float* addend,
                         int64_t ld_add, int act, float act_slope, float* out, int64_t ld_out, float* self_out, int64_t ld_self,
                         int out_node_major, void* stream);
/* mlg_sage_rank1_fwd_rows / mlg_sage_rank1_bwd_rows with NODE-MAJOR activation / gradient rows ((replica b, node i) at
 * i * replicas + b: a gene's replica rows are one contiguous block); arguments as the graph-major entries. */
int mlg_sage_rank1_fwd_rows_nm(const float* xs_t, const float* e_self, int64_t ld_self, const float* e_nbr, int64_t ld_nbr,
                               const int32_t* rowptr, const int32_t* idx, const float* val, const int32_t* order, int64_t n_rows,
                               int64_t C, int64_t replicas, const float* bias, float slope, float* out, int64_t ld_out,
                               uint64_t* mask_bits, void* stream);
int mlg_sage_rank1_bwd_rows_nm(const float* gz, int64_t ld_g, const float* y, const uint64_t* mask_bits, float slope, const float* xs,
                               int xs_transposed, const int32_t* rowptr, const int32_t* idx, const float* val,
                               const int32_t* order, int64_t n_rows, int64_t C, int64_t replicas, float* h, float* g_self,
                               int64_t ld_self, float* g_bias_rows, void* stream);

/* Fully factored first SAGE layer of MultilevelGNN (models/multilevel_gnn.py:150-151 feeding SAGEConv,
 * gcn_lib/sparse/torch_vertex.py:269-294).  The layer input x0[b,n,:] = x[b,n] * node_embedding[n,:] is rank-1 per node,
 * so both halves of the update  z = [x0 | mean_j(w_ij x0_j)] [W1 | W2 W_r]^T + bias  factor through two per-gene tables
 * E_self = emb W1^T and E_nbr = emb (W2 W_r)^T ([n_rows, C], C = Cout):
 *     out[b*n_rows+i,:] = LeakyReLU_slope( xs[b*n_rows+i] * e_self[i,:]
 *                                          + (1/cnt_i) * sum_{q in row i} val[q] * xs[b*n_rows+idx[q]] * e_nbr[idx[q],:] + bias )
 * (cnt_i = row length incl. the added self loop: PyG mean aggregation; bias NULL ok; slope 0 = ReLU).
 * Neither x0, the [x0 | agg] buffer nor the (replicas*n_rows)-row update GEMM are ever formed.  replicas >= 2, C % 4 == 0,
 * 16-byte aligned tables / out with leading dimensions that are multiples of 4; CSR / order as in mlg_gather_sum. */
int mlg_sage_rank1_fwd(const float* xs, const float* e_self, int64_t ld_self, const float* e_nbr, int64_t ld_nbr,
                       const int32_t* rowptr, const int32_t* idx, const float* val, const int32_t* order, int64_t n_rows,
                       int64_t C, int64_t replicas, const float* bias, float slope, float* out, int64_t ld_out,
                       uint64_t* mask_bits, void* stream);
/* mask_bits (NULL ok; C == 64 only): [n_rows][replicas] 64-bit words, bit 16*(c % 4) + c / 4 = (out[b,i,c] > 0): lets the
 * backward pass apply LeakyReLU' from 8 bytes per (row, replica) instead of re-reading the activation. */
/* Its backward w.r.t. the tables and the bias from gz = dL/dz [replicas*n_rows, C], one pass over the by-source CSR
 * (rowptr_t / idx_t / val_t / order_t; inv_cnt[i] = 1/cnt_i of the forward rows, NULL = 1):
 *     g_e12_parts[s*n_rows+j, 0:C]  = sum_{b in slice s} xs[b,j] * gz[b,j,:]                                       -> g_E_self
 *     g_e12_parts[s*n_rows+j, C:2C] = sum_{b in slice s} xs[b,j] * sum_{i: j in row i} val_ij * inv_cnt[i] * gz[b,i,:] -> g_E_nbr
 *     g_bias_parts[s*n_rows+j, :]   = sum_{b in slice s} gz[b,j,:]
 * for s < mlg_gather_sum_slices(n_rows, C, replicas); the caller adds the slices (fixed order: deterministic). */
int mlg_sage_rank1_bwd(const float* gz, int64_t ld_g, const float* xs, const int32_t* rowptr_t, const int32_t* idx_t,
                       const float* val_t, const float* inv_cnt, const int32_t* order_t, int64_t n_rows, int64_t C,
                       int64_t replicas, float* g_e12_parts, float* g_bias_parts, void* stream);

/* The same gradients organised by TARGET row so that gz is read exactly once (C == 32 or 64; forward CSR rowptr / idx /
 * val / order): per entry q of row i (source j = idx[q])  h[q,:] = (val[q] / cnt_i) * sum_b xs[b,j] * gz[b,i,:], and per row
 * g_self[i,:] = sum_b xs[b,i] * gz[b,i,:] (-> g_E_self, leading dimension ld_self), g_bias_rows[i,:] = sum_b gz[b,i,:].
 * g_E_nbr[j,:] = sum_{q: idx[q] == j} h[q,:] is a segment sum the caller runs over the by-source CSR with mlg_gather_sum
 * (single graph, idx = by-source position -> forward position).  h must hold rowptr[n_rows] rows of C floats.
 * y != NULL: gz is dL/dy of the layer's LeakyReLU(slope) output y (same layout as gz) and the kernel multiplies by the
 * activation derivative while loading (no separate activation-backward pass); mask_bits != NULL (C == 64): the same
 * from the sign bits mlg_sage_rank1_fwd wrote (y is then not read).  xs_transposed != 0: xs is [n_rows, replicas]. */
int mlg_sage_rank1_bwd_rows_supported(int64_t C);
int mlg_sage_rank1_bwd_rows(const float* gz, int64_t ld_g, const float* y, const uint64_t* mask_bits, float slope, const float* xs, int xs_transposed, const int32_t* rowptr, const int32_t* idx,
                            const float* val, const int32_t* order, int64_t n_rows, int64_t C, int64_t replicas, float* h,
                            float* g_self, int64_t ld_self, float* g_bias_rows, void* stream);

/* The forward pass with one WARP per gene for all replicas (C == 32 or 64): the neighbour's table row and its replica values
 * are loaded once per CSR entry.  xs_t [n_rows, replicas]: the node values TRANSPOSED (mlg_transpose_bn of xs [replicas,
 * n_rows]); the same matrix serves mlg_sage_rank1_bwd_rows (xs_transposed = 1).  Other arguments as mlg_sage_rank1_fwd;
 * tables / out 8-byte aligned with even leading dimensions. */
int mlg_transpose_bn(const float* xs, int64_t B, int64_t n, float* xs_t, void* stream);
int mlg_sage_rank1_fwd_rows_supported(int64_t C);
int mlg_sage_rank1_fwd_rows(const float* xs_t, const float* e_self, int64_t ld_self, const float* e_nbr, int64_t ld_nbr,
                            const int32_t* rowptr, const int32_t* idx, const float* val, const int32_t* order, int64_t n_rows,
                            int64_t C, int64_t replicas, const float* bias, float slope, float* out, int64_t ld_out,
                            uint64_t* mask_bits, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Tall-skinny transposed product: out[M,K] = A[rows,M]^T * X[rows,K], colsum[M] = sum_r A[r,:] (NULL ok).
 * The weight / bias gradient of the Linear layers on the path (SAGEConv.update's MLP and lin_r,
 * torch_vertex.py:281-291) where rows = B*N nodes and M, K <= 128.  fp32 FMA, fixed reduction order.
 * 16-byte aligned operands with M, K, ld_a, ld_x multiples of 4 take the 128-bit path.  workspace >= mlg_xty_workspace_bytes().
 */
int64_t mlg_xty_workspace_bytes(int64_t rows, int64_t M, int64_t K);
int mlg_xty(const float* A, int64_t ld_a, const float* X, int64_t ld_x, int64_t rows, int64_t M, int64_t K,
            float* out, float* colsum, void* workspace, int64_t workspace_bytes, void* stream);

/* The same product on the tensor cores (tcgen05, 3xTF32 split: fp32-accurate, relative error ~2^-20) for the shapes
 * that dominate the training step: K == 128 (X is [x | agg_x] of a 64-wide SAGE layer, or a 128-wide GENConv edge
 * encoder input), 16 <= M <= 128, M % 16 == 0, 16-byte aligned operands, ld multiples of 4.  Each 32-row chunk is
 * transposed + split in shared memory; per-CTA partial sums are reduced in a fixed order (deterministic). */
int mlg_xty_tc_supported(int64_t rows, int64_t M, int64_t K);
int64_t mlg_xty_tc_workspace_bytes(int64_t M);
int mlg_xty_tc(const float* A, int64_t ld_a, const float* X, int64_t ld_x, int64_t rows, int64_t M, int64_t K,
               float* out, float* colsum, float* colsum_x, void* workspace, int64_t workspace_bytes, void* stream);
/* (colsum_x [128]: column sums of X, NULL ok -- the bias gradient when the roles of A and X are swapped for a 128-wide
 *  output, e.g. the weight gradient of Linear(256 -> 128)) */

/* Weight folding of the fused SAGE layer (SAGEConv, torch_vertex.py:279-291: nn(cat[x, mean_j lin_r(x_j)]) with lin_r
 * commuted past the mean).  nn_w = nn.weight [cout, cin + r], lin_r_w = lin_r.weight [r, cin].
 * fwd: wcat = [W1 | W2 * W_r] [cout, 2cin], its 3xTF32 hi/lo split, and the hi/lo split of wcat^T [2cin, cout].
 * bwd: g_nn_w = [g_wcat[:, :cin] | g_wcat[:, cin:] * W_r^T],  g_lin_r_w = W2^T * g_wcat[:, cin:]. */
int mlg_sage_fold_fwd(const float* nn_w, const float* lin_r_w, int64_t cout, int64_t cin, int64_t r, float* wcat, float* wcat_hi,
                      float* wcat_lo, float* wcat_t_hi, float* wcat_t_lo, void* stream);
int mlg_sage_fold_bwd(const float* g_wcat, const float* nn_w, const float* lin_r_w, int64_t cout, int64_t cin, int64_t r,
                      float* g_nn_w, float* g_lin_r_w, void* stream);
/* The same folding in the STACKED layout the transform-first layer and the factored first layer use
 * (z = U + mean_j(w_ij V_j), [U | V] = x Wst^T + [b | 0]):  wst = [W1 ; W2 * W_r] [2cout, cin], its 3xTF32 split, the split
 * of wst^T [cin, 2cout] (dX GEMM) and bias2 = [nn_b | 0] [2cout] (NULL ok; nn_b NULL ok = zeros) in ONE launch.
 * bwd: g_wst [2cout, cin] with leading dimension ld, optionally the sum of two addends (g_wst_add NULL ok):
 * g_nn_w = [g_wst[:cout] | g_wst[cout:] * W_r^T],  g_lin_r_w = W2^T * g_wst[cout:]. */
int mlg_sage_fold_stacked_fwd(const float* nn_w, const float* lin_r_w, const float* nn_b, int64_t cout, int64_t cin, int64_t r,
                              float* wst, float* wst_hi, float* wst_lo, float* wst_t_hi, float* wst_t_lo, float* bias2,
                              void* stream);
int mlg_sage_fold_stacked_bwd(const float* g_wst, const float* g_wst_add, int64_t ld, const float* nn_w, const float* lin_r_w,
                              int64_t cout, int64_t cin, int64_t r, float* g_nn_w, float* g_lin_r_w, void* stream);

/* Pathway-wise independence term of MultilevelGNN.get_feature_loss (models/multilevel_gnn.py:336-346; no gradient, the
 * reference reads .data):  out[0] = (1 / (P(P-1)/2)) * sum_{i < P-1} mean_s | sum_g w_gi w_gL | / (sqrt(sum_g w_gi^2 *
 * sum_g w_gL^2) + 1e-7),  L = P-1, w = w_raw * mask (mask [G] or NULL), g over the genes of pathway segment s =
 * [segptr[s], segptr[s+1]) (genes sorted by segment).  Fixed summation order.  2 <= P <= 8; workspace: nseg floats. */
int mlg_pca_indep_loss(const float* w, const float* mask, const int32_t* segptr, int64_t nseg, int64_t P, float* out,
                       float* workspace, void* stream);

/* Head max-pool over a channel-LAST activation (nn.MaxPool2d((kh, kw)), stride = kernel, floor mode, of
 * multilevel_gnn.py:286): x_cl [B, H, W, C] in memory -> out_nchw [B, C, H/kh, W/kw] (the order flatten() expects) and the
 * window position of each maximum (first maximum in row-major scan order, ATen's tie rule).  Backward scatters g_out to
 * those positions and zero-fills the rest of g_x_cl [B, H, W, C]. */
int mlg_maxpool_cl_fwd(const float* x_cl, int64_t B, int64_t H, int64_t W, int64_t C, int64_t kh, int64_t kw,
                       float* out_nchw, uint8_t* argmax, void* stream);
int mlg_maxpool_cl_bwd(const float* g_out_nchw, const uint8_t* argmax, int64_t B, int64_t H, int64_t W, int64_t C,
                       int64_t kh, int64_t kw, float* g_x_cl, void* stream);

/* LayerNorm over the channel axis of a tall [rows, C] fp32 activation (nn.LayerNorm(C), biased variance): DeeperGCN's
 * res+ block norm (models/deepergcn.py:262-275) and the norm inside GENConv's MLP (gcn_lib/sparse/torch_nn.py:55-73).
 * C in {128, 256, 384, 512}; gamma / beta may be NULL (= 1 / 0).  fwd also writes the per-row mean and 1/std that bwd
 * reads; bwd writes the input gradient and (fixed summation order) the gamma / beta gradients (either may be NULL).
 * workspace >= mlg_layernorm_bwd_workspace_bytes(rows, C). */
int mlg_layernorm_supported(int64_t C);
int64_t mlg_layernorm_bwd_workspace_bytes(int64_t rows, int64_t C);
int mlg_layernorm_fwd(const float* x, const float* gamma, const float* beta, int64_t rows, int64_t C, float eps, float* y,
                      float* mean, float* rstd, void* stream);
int mlg_layernorm_bwd(const float* x, const float* g, const float* gamma, const float* mean, const float* rstd,
                      int64_t rows, int64_t C, float* gx, float* dgamma, float* dbeta, void* workspace,
                      int64_t workspace_bytes, void* stream);
/* The same norm followed by ReLU in one pass each way (deepergcn.py:268-270 `F.relu(norm(h))`, torch_nn.py MLP
 * Lin -> norm -> act): y = max(LN(x), 0); bwd masks g where the output was not positive (rebuilt from xhat, gamma, beta). */
int mlg_layernorm_relu_fwd(const float* x, const float* gamma, const float* beta, int64_t rows, int64_t C, float eps,
                           float* y, float* mean, float* rstd, void* stream);
int mlg_layernorm_relu_bwd(const float* x, const float* g, const float* gamma, const float* beta, const float* mean,
                           const float* rstd, int64_t rows, int64_t C, float* gx, float* dgamma, float* dbeta,
                           void* workspace, int64_t workspace_bytes, void* stream);

/* GENConv aggregation with a rank-1 AFFINE edge term: message_ij = relu(x_j + a_e * p + q) + eps, a_e = edge_scalar[e]
 * (one number per edge), p = edge_p, q = edge_q ([H]).  Same semantics, epilogues and outputs as mlg_gen_aggr_fwd / _bwd
 * with e_ij = a_e * p + q, but the [E, H] edge embedding is never read or written: this is DeeperGCN's edge path when
 * the raw edge attribute is a scalar weight -- Linear(1 -> H) (models/deepergcn.py:209) followed by each GENConv's own
 * Linear(H -> H) edge encoder (gcn_lib/sparse/torch_vertex.py:76-77) is affine in a_e.  g_edge [E, H] (gradient w.r.t.
 * the edge term, original edge order) is still produced: the source-side pass (mlg_gather_sum over the by-source CSR)
 * consumes it. */
int mlg_gen_aggr_fwd_affine(const float* x, const float* edge_scalar, const float* edge_p, const float* edge_q,
                            const int32_t* rowptr, const int32_t* col, const int32_t* eid, int64_t n, int64_t H, int mode,
                            float t, const float* t_dev, float p, const float* p_dev, const float* y_dev, float eps,
                            int epilogue, const float* msg_scale_dev, float* m, float* aux, float* h, void* stream);
/* g_p / g_q (both NULL ok): gradients of edge_p / edge_q, g_p = sum_e a_e * g_edge[e], g_q = sum_e g_edge[e], accumulated
 * inside the backward kernel (per-block partials in `workspace`, fixed-order two-level reduction) -- no second pass over
 * g_edge.  n_edges = rows of edge_scalar / g_edge.  workspace >= mlg_gen_aggr_bwd_affine_workspace_bytes(n, n_edges, H). */
int64_t mlg_gen_aggr_bwd_affine_workspace_bytes(int64_t n, int64_t n_edges, int64_t H);
int mlg_gen_aggr_bwd_affine(const float* g, const float* x, const float* edge_scalar, const float* edge_p,
                            const float* edge_q, const int32_t* rowptr, const int32_t* col, const int32_t* eid, int64_t n,
                            int64_t n_edges, int64_t H, int mode, int learn, float t, const float* t_dev, float p,
                            const float* p_dev, const float* y_dev, float eps, int epilogue, const float* msg_scale_dev,
                            const float* m, const float* aux, float* g_edge, float* g_x, float* partials, float* g_p,
                            float* g_q, void* workspace, int64_t workspace_bytes, void* stream);
/* mlg_gen_aggr_bwd_affine with the source-side sum inside the kernel (see mlg_gen_aggr_bwd_src; same support query; needs
 * g_p / g_q either both NULL or the fused per-block sums, i.e. H <= 256): g_edge may be NULL -- then no [E,H] tensor is
 * written at all. */
int mlg_gen_aggr_bwd_affine_src(const float* g, const float* x, const float* edge_scalar, const float* edge_p,
                                const float* edge_q, const int32_t* rowptr, const int32_t* col, const int32_t* eid, int64_t n,
                                int64_t n_edges, int64_t H, int mode, int learn, float t, const float* t_dev, float p,
                                const float* p_dev, const float* y_dev, float eps, int epilogue, const float* msg_scale_dev,
                                const float* m, const float* aux, float* g_edge, float* g_x, float* partials, float* g_p,
                                float* g_q, void* workspace, int64_t workspace_bytes, void* stream);
/* Weighted column sums of a tall matrix: u[c] = sum_r a[r] * G[r,c] (u NULL ok), v[c] = sum_r G[r,c] (v NULL ok); one
 * streaming pass, fixed summation order.  C % 4 == 0, C <= 1024.  workspace >= mlg_wcolsum_workspace_bytes(rows, C). */
int64_t mlg_wcolsum_workspace_bytes(int64_t rows, int64_t C);
int mlg_wcolsum(const float* G, int64_t ld, const float* a, int64_t rows, int64_t C, float* u, float* v, void* workspace,
                int64_t workspace_bytes, void* stream);

/* Metrics of an evaluation split (train.py:71-109 of the reference), one kernel after a 32-byte memset of the workspace:
 * out[0] = torch.nn.BCELoss(weight) of pred [n,2] against y [n,2] (mean over the 2n elements, logs clamped at -100, weight =
 * the class row class_w [2], NULL = 1); out[1] = accuracy of argmax(pred) against argmax(y) (ties -> index 0, NaN is the
 * maximum, as torch.argmax); out[2] = ROC AUC of pred[:,1] for the labels argmax(y), exactly: the Mann-Whitney count (2 per
 * positive/negative pair with s_pos > s_neg, 1 per tie) in 64-bit integers over 2 P N -- NaN when one class is absent.
 * Deterministic (integer atomics, fixed-order BCE sum): bit-identical results for the same inputs.  1 <= n <= 65 536
 * (O(n^2) pair count).  workspace (8-byte aligned) >= mlg_eval_metrics_workspace_bytes(n). */
int64_t mlg_eval_metrics_workspace_bytes(int64_t n);
int mlg_eval_metrics(const float* pred, const float* y, int64_t n, const float* class_w, float* out, void* ws,
                     int64_t ws_bytes, void* stream);

/* Skinny Linear forward: out[rows,N] = act(x[rows,K] * W[N,K]^T + bias), rows <= 32, any K (long reduction).
 * MultilevelGNN's head Linear(6913 -> 256) on a batch of <= 32 graphs (models/multilevel_gnn.py:104-110): a batched
 * GEMV bound by the one pass over W.  act: 0 none, 1 LeakyReLU(slope) (slope 0 = ReLU).  fp32 FMA, fixed summation
 * order.  workspace >= mlg_skinny_linear_workspace_bytes(N, K). */
int64_t mlg_skinny_linear_workspace_bytes(int64_t N, int64_t K);
int mlg_skinny_linear(const float* x, int64_t ld_x, const float* W, int64_t ld_w, const float* bias, int64_t rows,
                      int64_t N, int64_t K, int act, float slope, float* out, int64_t ld_out, void* workspace,
                      int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * MultilevelGNN's classification head + loss, fused (models/multilevel_gnn.py:262-290; train.py:60,118).
 * Replaces: Conv2d(32->32,1x1)+ReLU, Conv2d(32->64,1x1)+ReLU, MaxPool2d((kh,kw)) (stride = kernel, floor mode), Dropout,
 * flatten, cat(age), Linear(K->D)+ReLU+Dropout, Linear(D->2), Softmax, BCELoss(weight) and their backward ops.
 *
 * x_cl [B,H,W,32]: the pooled pathway features, channel-last (mlg_pool_fwd's layout).  a0 [B, ld]: the flattened head
 * input in NCHW order (column c*Ho*Wo + ho*Wo + wo, c < 64) and, when age != NULL, age[b] in column 64*Ho*Wo.
 * Dropout: element kept iff drop_bits[i] >= p * 2^31 and scaled by 1/(1-p); drop_bits are caller-provided uniform
 * int32 words in [0, 2^31) (NULL / p == 0: no dropout) indexed like the tensor they mask ([B, 64*Ho*Wo] and [R, D]).
 * Backward of conv/pool recomputes both convolutions; the gradient of a window goes to its FIRST maximum (ATen).
 * g_x_cl [B,H,W,32] is fully written (zeros for pixels the floor-mode pool drops). */
int mlg_head_conv_pool_supported(int64_t cin, int64_t c1, int64_t c2);
int64_t mlg_head_conv_pool_bwd_workspace_bytes(int64_t B, int64_t H, int64_t W, int64_t kh, int64_t kw);
int mlg_head_conv_pool_fwd(const float* x_cl, const float* W1, const float* b1, const float* W2, const float* b2,
                           const float* age, const int32_t* drop_bits, float drop_p, int64_t B, int64_t H, int64_t W,
                           int64_t kh, int64_t kw, float* a0, int64_t ld, void* stream);
int mlg_head_conv_pool_bwd(const float* g_a0, int64_t ld, const float* x_cl, const float* W1, const float* b1,
                           const float* W2, const float* b2, const int32_t* drop_bits, float drop_p, int64_t B, int64_t H,
                           int64_t W, int64_t kh, int64_t kw, float* g_x_cl, float* g_W1, float* g_b1, float* g_W2,
                           float* g_b2, void* workspace, int64_t workspace_bytes, void* stream);
/* a1 [R,D] = dropout(relu(a0[:, :K] W0^T + b0)); pred [R,2] = softmax(a1 W3^T + b3); with y [R,2] given also
 * loss[0] = mean(weight * BCE(pred, y)) (weight [R,2] or NULL; logs clamped at -100 like ATen).  R <= 64.
 * Backward: g_pred [R,2] and / or g_loss [1] (device scalars) -> g_a0 [R, ld_g] (NULL: not needed), g_W0 [D,K], g_b0,
 * g_W3 [2,D], g_b3; D a multiple of 32 up to 512. */
int64_t mlg_head_mlp_workspace_bytes(int64_t R, int64_t D, int64_t K);
int mlg_head_mlp_fwd(const float* a0, int64_t ld_a, const float* W0, const float* b0, const float* W3, const float* b3,
                     const int32_t* drop_bits, float drop_p, const float* y, const float* weight, int64_t R, int64_t D,
                     int64_t K, float* a1, float* pred, float* loss, void* workspace, int64_t workspace_bytes, void* stream);
/* Input-gradient-only mode of both head backward calls: pass NULL for all four weight-gradient outputs (and, for
 * mlg_head_conv_pool_bwd, a NULL workspace).  The kernels then skip the weight-gradient products: mlg_head_mlp_bwd reads
 * W0 once for g_a0 and never stages the gW0 slice, mlg_head_conv_pool_bwd skips its per-block partials and their reduce.
 * With non-NULL outputs both calls run exactly as before. */
int mlg_head_mlp_bwd(const float* g_pred, const float* g_loss, const float* pred, const float* y, const float* weight,
                     const float* a0, int64_t ld_a, const float* a1, const float* W0, const float* W3, float drop_p,
                     int64_t R, int64_t D, int64_t K, float* g_a0, int64_t ld_g, float* g_W0, float* g_b0, float* g_W3,
                     float* g_b3, void* stream);

/* ---------------------------------------------------------------------------------------------
 * DiffPool at the reference's size, fused (models/diff_pooling.py:59-65,116-133 with PyG DenseSAGEConv(normalize=True)
 * and dense_diff_pool; called from VAE.predict_head, models/vae.py:238-243): one persistent CTA per sample keeps the
 * whole sample in shared memory.  1 or 2 pooling layers, after_pooling_layer = 1, shared adjacency adj [n0, n0].
 *   dims: HOST array, 4 per layer: (n nodes, c in-channels, k clusters, h embedding channels); layer 1 = (k0, h0, k1, h1)
 *   weights: HOST array of 9 DEVICE pointers per layer:
 *            gnn_pool (lin_rel.weight [k,c], lin_root.weight [k,c], lin_root.bias [k]),
 *            gnn_embed (lin_rel.weight [h,c], lin_root.weight [h,c], lin_root.bias [h]),
 *            after_pool (lin_rel.weight [h,h], lin_root.weight [h,h], lin_root.bias [h])
 *   out [b, k_last, h_last]; stats [b, 2*layers] = per sample and layer (||adj_l - S S^T||_F^2, sum_rows sum_k -S log(S+1e-15)):
 *   link = sum_l sqrt(sum_b F_l) / numel(adj_l), entropy = sum_l sum_b E_l / (b n_l) are formed by the caller.
 * Backward: g_out [b, k_last, h_last]; coef DEVICE [2*layers] = per layer (g_link / (sqrt(sum_b F_l) numel(adj_l)),
 *   g_entropy / (b n_l)); g_x [b, n0, c0]; g_weights: ONE device buffer of mlg_diffpool_grad_floats floats, the 9 gradients
 *   of each layer back to back in the order of `weights`; workspace >= mlg_diffpool_ctas(b) * grad_floats * 4 bytes.
 *   state (16-byte aligned DEVICE buffer of b * mlg_diffpool_state_floats floats, or NULL): the forward intermediates
 *   backward reads again.  Forward writes it when given; backward given the same buffer skips recomputing the forward pass
 *   (NULL: it recomputes).
 * mlg_diffpool_supported: the per-sample working set fits the 227 KB of shared memory of one SM. */
int64_t mlg_diffpool_smem_bytes(int64_t layers, const int64_t* dims);
int mlg_diffpool_supported(int64_t layers, const int64_t* dims);
int64_t mlg_diffpool_grad_floats(int64_t layers, const int64_t* dims);
int64_t mlg_diffpool_state_floats(int64_t layers, const int64_t* dims);
int64_t mlg_diffpool_ctas(int64_t b);
int mlg_diffpool_fwd(const float* x, const float* adj, const float* const* weights, int64_t layers, const int64_t* dims,
                     int64_t b, float* out, float* stats, float* state, void* stream);
int mlg_diffpool_bwd(const float* g_out, const float* coef, const float* x, const float* adj, const float* const* weights,
                     int64_t layers, const int64_t* dims, int64_t b, float* g_x, float* g_weights, const float* state,
                     void* workspace, int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Per-pathway decoders of the VAE, grouped (models/vae.py:54-74 builds one Linear(F, D_i)-ReLU-Linear(D_i, n_i) block per
 * pathway, foreach_decoder :216-222 runs them on h[:, i, :] and concatenates): one CTA per pathway, one launch per row chunk.
 *   x [B, S, F]; packed: all blocks' parameters in one DEVICE buffer; table: DEVICE int64 [S, 8], per pathway the float offsets
 *   into `packed` of (W1 [D,F], b1 [D], W2 [n,D], b2 [n]) and (D, n, first output column, first hidden column);
 *   Dmax = max_i D_i; out [B, total_out] (total_out = sum n_i); h_saved [B, total_hidden] (sum D_i) = post-ReLU activations,
 *   written by forward when non-NULL and required by backward.
 * Backward: g_out [B, total_out] -> g_x [B, S, F] (NULL: not needed) and g_packed (same layout as packed; only the
 *   parameter elements are written, one writer each -- gaps between arrays are left untouched).
 * mlg_decoder_max_rows: batch rows one launch holds in shared memory; larger B is processed in chunks internally. */
int64_t mlg_decoder_max_rows(int64_t F, int64_t Dmax, int backward);
int mlg_decoder_fwd(const float* x, const float* packed, const int64_t* table, int64_t B, int64_t S, int64_t F,
                    int64_t Dmax, int64_t total_out, int64_t total_hidden, float* out, float* h_saved, void* stream);
int mlg_decoder_bwd(const float* g_out, const float* x, const float* h_saved, const float* packed, const int64_t* table,
                    int64_t B, int64_t S, int64_t F, int64_t Dmax, int64_t total_out, int64_t total_hidden, float* g_x,
                    float* g_packed, void* stream);

/* z[r,c] = LeakyReLU_slope(z[r,c] + bias[c]) in place (bias NULL ok; slope 0 = ReLU): the bias + activation
 * of SAGEConv.update's MLP (torch_vertex.py:288-291) after the update GEMM. */
int mlg_bias_act(float* z, const float* bias, int64_t rows, int64_t C, float slope, void* stream);

/* ---------------------------------------------------------------------------------------------
 * MultilevelGNN prologue: x0[b*N+n, :] = xs[b*N+n] * emb[n, :]   (models/multilevel_gnn.py:150-151)
 * and its backward g_emb[n,:] = sum_b xs[b,n] * g_x0[b,n,:].
 */
int mlg_embed_scale_fwd(const float* xs, const float* emb, int64_t B, int64_t N, int64_t C, float* out,
                        void* stream);
int mlg_embed_scale_bwd(const float* xs, const float* g_out, int64_t B, int64_t N, int64_t C,
                        float* g_emb, void* stream);
/* Gradient w.r.t. the node values of the same prologue: g_xs[b*N+n] = <g_out[b*N+n, :], emb[n, :]>  (g_xs [B*N]). */
int mlg_embed_scale_bwd_xs(const float* g_out, const float* emb, int64_t B, int64_t N, int64_t C, float* g_xs, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Gradient w.r.t. the node values xs [B*N] of the fully factored first SAGE layer (mlg_sage_rank1_fwd_rows):
 *     g_xs[b,j] = <gz[b,j,:], E_self[j,:]> + sum_{(i,q): idx_q = j} (val_q / cnt_i) <gz[b,i,:], E_nbr[j,:]>
 * gz [B*n_rows, C] (ld_g) is dL/dz or, with mask_bits (C == 64, the forward's sign bits) or y (the layer output, layout of
 * gz) given, dL/dy; gz_node_major: its rows are (replica b, node i) at i * B + b.  rowptr / idx / val / order: the
 * forward (by-target) CSR as for the forward call (cap entries); rowptr_t / fwd_pos_t: the by-source CSR whose entries
 * are positions in the forward CSR (Topology.bwd.rowptr, Topology.bwd2fwd).  g_xs [B*n_rows] graph-major.  C == 32 or
 * 64, 1 <= replicas <= 64.  Per-entry values ([cap, B]) and self terms ([n_rows, B]) go to the workspace; the segment sum
 * runs in a fixed order: bit-identical results from run to run. */
int64_t mlg_sage_rank1_bwd_xs_workspace_bytes(int64_t cap, int64_t n_rows, int64_t replicas);
int mlg_sage_rank1_bwd_xs(const float* gz, int64_t ld_g, int gz_node_major, const float* y, const uint64_t* mask_bits,
                          float slope, const float* e_self, int64_t ld_self, const float* e_nbr, int64_t ld_nbr,
                          const int32_t* rowptr, const int32_t* idx, const float* val, const int32_t* order,
                          const int32_t* rowptr_t, const int32_t* fwd_pos_t, int64_t n_rows, int64_t cap, int64_t C,
                          int64_t replicas, float* g_xs, void* workspace, int64_t workspace_bytes, void* stream);

/* acc[p, c] = (accumulate ? acc[p, c] : 0) + sum_{s = slot_ptr[p]}^{slot_ptr[p+1]-1} w[s] * g[s * ld_g + c],  c < N:
 * per-slot gradients summed into per-output rows in slot order (integrated gradients' trapezoid sum, also across
 * replays).  acc [n_out, N], slot_ptr int32 [n_out + 1]. */
int mlg_attr_accumulate(const float* g, int64_t ld_g, const float* w, const int32_t* slot_ptr, int64_t n_out, int64_t N,
                        int accumulate, float* acc, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Gene -> pathway pool (models/multilevel_gnn.py:205-239): value mask, gather by gene_pca_match,
 * missing-gene mask, per-gene projection, segment sum -- without materialising [B,C,G,P].
 *     out[b,c,s,p] = sum_{g in seg(b,s)} vm[node] * x[node, c] * w[g,p],  node = b*N + match[b,g] (skipped if < 0)
 * seg_rowptr int32 [B*S+1], seg_slot int32 [B*G] : CSR of slots (b*G+g) grouped by (b*S + raw_indice[b,g])
 *   (built with mlg_csr_build on edge_index = [slot; segment]).
 * x [B*N, C]; vm [B*N] or NULL (value_att_mask multiplier, batch.x); match int64 [B,G];
 * w [G,P] = learnable_pca_params * info_mask (caller multiplies, G*P elements);
 * out_cl [B, S, P, C]: CHANNEL-LAST; the reference's [B, C, 146, 3P] tensor is its permute(0,3,1,2) view
 * (s = pathway*3 + omic, so (omic, p) merge into the reference's last axis without a copy).
 * wrap_negative != 0 reproduces python negative indexing when pca_match_mask is False.
 */
int mlg_pool_fwd(const float* x, const float* vm, const int64_t* match, const float* w,
                 const int32_t* seg_rowptr, const int32_t* seg_slot, int64_t B, int64_t N, int64_t C,
                 int64_t G, int64_t S, int64_t P, int wrap_negative, float* out_cl, void* stream);

/* Backward.  g_out_cl [B,S,P,C] = gradient of out_cl (channel-last).
 * mlg_pool_bwd_x: g_x [B*N, C] via the node-side CSR (slots grouped by the node they read, built with
 *   mlg_csr_build on [slot; node]).  replicas == 1: node_rowptr [B*N+1], node_slot [B*G], seg_of_slot int32
 *   [B*G] = b*S + raw_indice[b,g].  replicas == B: gene_pca_match / raw_indice are identical for all graphs
 *   (multiloader.py:697) and the CSR covers ONE graph: node_rowptr [N+1], node_slot [G], seg_of_slot [G] in [0,S).
 * mlg_pool_bwd_w: g_w [G,P] (gradient w.r.t. the masked product w; caller multiplies by info_mask). */
int mlg_pool_bwd_x(const float* g_out_cl, const float* vm, const float* w, const int32_t* node_rowptr,
                   const int32_t* node_slot, const int32_t* seg_of_slot, int64_t B, int64_t N, int64_t C,
                   int64_t G, int64_t S, int64_t P, int64_t replicas, float* g_x, void* stream);
int mlg_pool_bwd_w(const float* g_out_cl, const float* x, const float* vm, const int64_t* match,
                   const int64_t* raw_indice, int64_t B, int64_t N, int64_t C, int64_t G, int64_t S,
                   int64_t P, int wrap_negative, int64_t replicas, float* g_w, void* stream);
/* Both gradients in ONE pass over the node-side CSR (x streamed in node order, every g_out_cl row loaded once):
 * g_x as above; per-graph partial weight gradients go to workspace [B*G*P] floats and are reduced over the
 * graphs in a fixed order into g_w.  C <= 128.  Node-side structures as for mlg_pool_bwd_x.
 * mask_input != 0: g_x *= (x > 0 ? 1 : mask_slope), the derivative of the (Leaky)ReLU that produced x (the last GNN
 * layer's output), so that layer receives dL/dz directly and skips its own activation-backward pass.
 * w_mask [G] (or NULL): w was params * w_mask[g] (info_mask, multilevel_gnn.py:222); g_w is then dL/dparams. */
int mlg_pool_bwd(const float* g_out_cl, const float* x, const float* vm, const float* w, const int32_t* node_rowptr,
                 const int32_t* node_slot, const int32_t* seg_of_slot, int64_t B, int64_t N, int64_t C, int64_t G,
                 int64_t S, int64_t P, int64_t replicas, float* g_x, float* g_w, float* workspace, int mask_input,
                 float mask_slope, const float* w_mask, void* stream);
/* mlg_pool_bwd with a choice of layout for g_x.  gx_node_major != 0 (C == 32, replicas == B > 1, see
 * mlg_pool_bwd_node_major_supported): the row of (graph b, node i) is i * B + b -- the B replica rows of a node are one
 * contiguous 128 * B-byte block, which is what the by-source aggregation consuming this gradient (mlg_gather_sum_nm)
 * gathers per CSR entry -- instead of b * N + i. */
int mlg_pool_bwd_node_major_supported(int64_t C, int64_t replicas);
int mlg_pool_bwd_layout(const float* g_out_cl, const float* x, const float* vm, const float* w, const int32_t* node_rowptr,
                        const int32_t* node_slot, const int32_t* seg_of_slot, int64_t B, int64_t N, int64_t C, int64_t G,
                        int64_t S, int64_t P, int64_t replicas, float* g_x, float* g_w, float* workspace, int mask_input,
                        float mask_slope, const float* w_mask, int gx_node_major, void* stream);
/* mlg_pool_bwd_layout that also returns the gradient w.r.t. the value mask vm (vm and g_vm [B*N] required):
 *     g_vm[b,n] = sum_c x[b,n,c] * u[b,n,c],   u[b,n,c] = sum_{slots of n} sum_p w[g,p] * g_out[b,seg,p,c]
 * (g_x = vm * u, times the activation derivative with mask_input), computed in the same pass as g_x -- never by dividing
 * g_x by vm.  g_w and workspace may be NULL: then no weight gradient is formed (the input-gradient-only backward);
 * g_x is always written, in the layout gx_node_major selects. */
int mlg_pool_bwd_vm(const float* g_out_cl, const float* x, const float* vm, const float* w, const int32_t* node_rowptr,
                    const int32_t* node_slot, const int32_t* seg_of_slot, int64_t B, int64_t N, int64_t C, int64_t G,
                    int64_t S, int64_t P, int64_t replicas, float* g_x, float* g_w, float* workspace, int mask_input,
                    float mask_slope, const float* w_mask, int gx_node_major, float* g_vm, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Dilated kNN graph (models/gcn_lib/sparse/torch_edge.py:53-104, dense/torch_edge.py:32-58):
 * fp32 distance d_ij = (|x_i|^2 + (-2 x_i.x_j)) + |x_j|^2, k*dilation nearest per point (self
 * included), ascending distance, ties by lowest index; every dilation-th rank is kept.
 * x [B, N, D]; out_nbr / out_ctr int64 [B*N*k] with per-graph node offsets (sparse layout, offset != 0)
 * or without (dense layout).  out_dist [B*N*k] optional (NULL ok).
 * workspace: mlg_knn_workspace_bytes(B, N, D, k, dilation) bytes.  With at least B*N*4 bytes (squared norms) the fp32
 * kernel runs; with the full amount, graphs of >= 4096 points (k*dilation <= 16, D <= 128) search their candidates on
 * the tensor cores (3xTF32) and re-evaluate / certify them in fp32 -- the output is identical to the fp32 kernel's.
 */
int64_t mlg_knn_workspace_bytes(int64_t B, int64_t N, int64_t D, int64_t k, int64_t dilation);
int mlg_knn_graph(const float* x, int64_t B, int64_t N, int64_t D, int64_t k, int64_t dilation,
                  int add_offset, int64_t* out_nbr, int64_t* out_ctr, float* out_dist, void* workspace,
                  int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Dense contractions of DiffPool (models/diff_pooling.py:61-64 -> PyG dense_diff_pool / DenseSAGEConv:
 * S^T.X, S^T.A.S, A.X, S.S^T) on the tcgen05 tensor cores:
 *     C[b][M,N] = alpha * A[b][M,K] . B[b][N,K]^T     A, B bf16 K-major (row-major [rows, K]); C fp32 row-major
 * TMA-fed 128B-swizzled tiles, accumulation in tensor memory (fp32).  lda/ldb multiples of 8 elements, operands
 * 16-byte aligned; stride_* are per-batch element strides (ignored for batch == 1).
 * mlg_cast_bf16 produces the K-major bf16 operands from fp32 row-major matrices [rows, cols]
 * (transpose != 0: dst[b][c][r] = src[b][r][c], i.e. dst is [cols, rows]).
 */
int mlg_cast_bf16(const float* src, int64_t ld_src, int64_t rows, int64_t cols, int64_t batch, int transpose,
                  void* dst_bf16, int64_t ld_dst, void* stream);
int mlg_gemm_bf16(const void* A, int64_t lda, int64_t stride_a, const void* B, int64_t ldb, int64_t stride_b,
                  float* C, int64_t ldc, int64_t stride_c, int64_t M, int64_t N, int64_t K, int64_t batch,
                  float alpha, void* stream);
/* Same product with a caller-owned workspace (mlg_gemm_bf16_workspace_bytes() bytes, 16-byte aligned, ZEROED ONCE when
 * it is allocated, one per stream): for M, N >= 256 a persistent stream-K grid of SM pairs splits the (tile, k block)
 * stream evenly, so products with fewer tiles than SM pairs (S^T.X) still fill the machine; partial tiles meet in the
 * workspace and are added in a fixed order (reproducible).  Other shapes fall through to mlg_gemm_bf16.  Replaces
 * the same torch.matmul call sites (PyG dense_diff_pool / DenseSAGEConv behind models/diff_pooling.py:61-64). */
int64_t mlg_gemm_bf16_workspace_bytes(void);
int mlg_gemm_bf16_ws(const void* A, int64_t lda, int64_t stride_a, const void* B, int64_t ldb, int64_t stride_b,
                     float* C, int64_t ldc, int64_t stride_c, int64_t M, int64_t N, int64_t K, int64_t batch,
                     float alpha, void* workspace, int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * fp32-accurate tall GEMM on the tensor cores (3xTF32 split, fp32 accumulation in tensor memory):
 *     C[M,N] = act( A[M,K] . B[N,K]^T + bias ),  act: 0 none, 1 LeakyReLU(slope) (slope 0 = ReLU)
 * for the Linear layers around the aggregations (SAGEConv.update MLP + lin_r, torch_vertex.py:281-291; GENConv
 * edge encoder, torch_vertex.py:76-77): M = nodes / edges (huge), 32 <= K <= 256 (K % 32 == 0), 16 <= N <= 256
 * (N % 16 == 0).  B_hi / B_lo [N,K] are the weight split by mlg_split_tf32 (hi = top 19 bits, lo = w - hi).
 * Relative error ~2^-20 (passes the fp32 rtol-1e-4 parity bar; plain TF32 would not).
 */
int mlg_split_tf32(const float* w, int64_t n, float* hi, float* lo, void* stream);
int mlg_gemm_tf32x3_supported(int64_t M, int64_t N, int64_t K);
int mlg_gemm_tf32x3(const float* A, int64_t lda, const float* B_hi, const float* B_lo, const float* bias, float* C,
                    int64_t ldc, int64_t M, int64_t N, int64_t K, int act, float slope, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Adam (torch.optim.Adam semantics, amsgrad off; train.py:112,66) over ONE flat fp32 buffer of parameters, their
 * gradients (the data-parallel gradient bucket) and the two moment buffers.  step_dev: device float holding the number
 * of steps taken so far (incremented by the call), so the update can be replayed inside a CUDA graph. */
int mlg_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* step_dev, int64_t n,
                  float lr, float beta1, float beta2, float eps, float weight_decay, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Data-parallel optimizer step over NVLink / NVSwitch peer memory: reduce-scatter(gradients) -> Adam on the owned
 * 1/world shard -> all-gather(parameters) as ONE kernel per rank, replacing "NCCL all-reduce + replicated Adam" of the
 * data-parallel wrapper around train.py:62-66 (the reference itself is single-device).  Every rank keeps its flat
 * gradient bucket, flat parameter buffer and a flag block (mlg_peer_flag_bytes(), zero-initialised) in device memory
 * from mlg_peer_alloc (cudaMalloc, zeroed) that the other ranks of the box map with mlg_peer_export / mlg_peer_open
 * (CUDA IPC, 64-byte handle).  peer_grads / peer_params / peer_flags are HOST arrays of `world` device pointers indexed
 * by rank (entry `rank` = this rank's own buffers).  [lo, hi): the CHUNK of the flat buffers this call updates (lo a multiple
 * of 4, hi - lo a multiple of 4*world; one flag block, one step counter and one optimizer-state shard PER CHUNK); rank r owns
 * the r-th 1/world of the chunk, and exp_avg / exp_avg_sq hold only that shard.  Chunks let the trainer update parameters
 * whose gradients are final early (the classifier head) on a forked branch while backward still runs.  Gradients are summed
 * in rank order and scaled by 1/world, so every rank ends with bitwise identical parameters.  step_dev as in mlg_adam_step.
 * The kernel synchronises the ranks itself (system-scope flags): every rank must issue the same sequence of calls.  A wait
 * longer than timeout_s (<= 0: 5 s) is a hard failure: the update is skipped (parameters and optimizer state untouched), the
 * status word of this rank AND of every peer is set (sticky: later calls return immediately; mlg_peer_status, 0 = ok) and,
 * when host_status != NULL (a pinned host int32, device-addressable), 1 is stored there so that the host can poll without a
 * device synchronisation.  max_blocks > 0 caps the grid (default 96 blocks of 512 threads) for a chunk that runs next to
 * other kernels.  Graph-capturable. */
int64_t mlg_peer_flag_bytes(void);
void* mlg_peer_alloc(int64_t bytes);
int mlg_peer_free(void* ptr);
int mlg_peer_export(void* ptr, void* handle64);
void* mlg_peer_open(const void* handle64);
int mlg_peer_close(void* ptr);
int mlg_peer_adam_step(const float* const* peer_grads, float* const* peer_params, void* const* peer_flags, int world,
                       int rank, int64_t lo, int64_t hi, float* exp_avg, float* exp_avg_sq, float* step_dev, float lr,
                       float beta1, float beta2, float eps, float weight_decay, double timeout_s, int32_t* host_status,
                       int max_blocks, void* stream);
/* Test support (one GPU): `world` ranks whose arenas all live on this device, stepped by ONE cooperative launch (blocks that
 * wait on one another must be co-resident).  exp_avg / exp_avg_sq / step_dev: HOST arrays of one device pointer per rank;
 * ranks_dev: device scratch of mlg_peer_emulated_bytes(world) bytes.  Synchronises the stream once (argument upload). */
int64_t mlg_peer_emulated_bytes(int world);
int mlg_peer_adam_step_emulated(const float* const* peer_grads, float* const* peer_params, void* const* peer_flags, int world,
                                int64_t lo, int64_t hi, float* const* exp_avg, float* const* exp_avg_sq, float* const* step_dev,
                                float lr, float beta1, float beta2, float eps, float weight_decay, double timeout_s,
                                void* ranks_dev, void* stream);
int mlg_peer_status(const void* flags, int* status_out);

#ifdef __cplusplus
}
#endif
#endif /* MLG_B200_H */
