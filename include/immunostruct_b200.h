/* immunostruct_b200 -- C ABI of the B200 (sm_100a) kernels behind the ImmunoStruct hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  The reference is pure
 * Python/PyTorch and has no FFI of its own; each entry point below names the reference call
 * (file:line under immunostruct/) whose GPU work it replaces.  The Python host layer
 * (immunostruct_b200/_C.py) binds these with ctypes; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (including scratch / partial buffers);
 *     launchers never allocate and never synchronise; work is enqueued on `stream` (a cudaStream_t);
 *   - return value: 0 = enqueued; < 0 = argument error (-1 bad argument, -2 unsupported size);
 *     > 0 = cudaError_t of the failed launch;
 *   - all floating tensors are fp32, row-major, contiguous unless a leading dimension is passed;
 *     graph ids are int64 at the reference-facing surface (DGL default) and int32 inside the CSR;
 *   - no floating-point atomics: results are bit-reproducible on a given device.
 */
#ifndef IMMUNOSTRUCT_B200_H
#define IMMUNOSTRUCT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- device / sizing queries ------------------------------------------------------------------ */
int is_num_sms(void);
int is_egnn_node_grid(int64_t n_nodes);       /* #partial blocks written by node_post_bwd / node_pre_bwd */
int is_egnn_edge_bwd_grid(int64_t n_nodes);   /* #partial blocks written by edge_bwd */
int is_attn_max_nodes(void);                  /* largest graph the attention kernels stage on chip */
int is_loss_num_partials(void);

/* ---- collation: dgl.batch (data/utils.py:163,169-170) + DGL's lazy dst-sorted CSC + its transpose.
 * scratch: int32[2*n_nodes]; stats: int32[4] = {max in-degree, #endpoints out of range,
 * max nodes per graph, #empty graphs}. */
int is_collate_csr(const int64_t* src_local, const int64_t* dst_local, const int64_t* node_counts,
                   const int64_t* edge_counts, int n_graphs, int64_t n_nodes, int64_t n_edges,
                   int64_t* node_off, int64_t* edge_off, int64_t* edge_index, int64_t* batch,
                   int* indptr, int* csr_src, int* csr_dst, int* csr_eid, int* outptr, int* csc_pos,
                   int* scratch, int* stats, void* stream);

/* ---- EGNNConv (dgl.nn.EGNNConv, models/hybrid_models.py:29-31,89-90; SURVEY Appendix A.3) --------
 * F = input feature width (20 for layer 0, 64 afterwards).  W1 = edge_mlp.0.weight [64, 2F+2],
 * W2/b2 = edge_mlp.2, W3/b3 = coord_mlp.0, w4 = coord_mlp.2.weight [1,64], W5/b5 = node_mlp.0
 * [64, F+64], W6/b6 = node_mlp.2.  PQ [n,128], hn [n,64]; status: int32 set to 1 if a node has
 * more than 128 in-edges (unsupported). */
int is_egnn_node_pre_fwd(const float* h, int64_t ldh, int F, const float* W1, const float* b1, float* PQ,
                         int64_t n_nodes, void* stream);
int is_egnn_edge_fwd(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                     const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                     const float* W1, int F, const float* W2, const float* b2,
                     const float* W3, const float* b3, const float* w4, int update_coords,
                     float* hn, float* x_out, int64_t n_nodes, int* status, void* stream);
/* tcgen05 / TMEM variant of is_egnn_edge_fwd: the two per-tile 128x64x64 GEMMs run on the tensor
 * cores.  precision 0 = bf16 operands (fp32 accumulate), 2 = 3xTF32, 3 = bf16x3, 4 = fp16x2 (fp16 hi / lo operand pairs,
 * inference forward only, activations beyond +-65504 overflow to inf) -- 2, 3, 4 are fp32-accurate;
 * fast_act != 0 selects the 5-instruction SiLU in the fp32-accurate modes (inference path). */
int is_egnn_edge_fwd_tc(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                        const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                        const float* W1, int F, const float* W2, const float* b2,
                        const float* W3, const float* b3, const float* w4, int update_coords, int precision,
                        int fast_act, float* hn, float* x_out, int64_t n_nodes, int* status, void* stream);
/* One whole EGNN layer of the fp16x2 inference forward in one launch (csrc/egnn_tc2.cu): is_egnn_edge_fwd_tc with precision 4
 * followed by is_egnn_node_post_pre_tc with precision 4, bit-identical.  Each CTA runs the node MLP and the next projections of
 * its own destination nodes once its edge tiles are done, so hn is written and read back within the launch.  h / ldh / F =
 * the layer's input features; update_coords 1 needs next_kind 1 (W1n = next edge_mlp.0.weight [64,130], PQn [n,128]);
 * update_coords 0 takes next_kind 2 (W1n = [Wq;Wk;Wv] [192,64], PQn = QKV [n,192]) or W1n / b1n / PQn NULL. */
int is_egnn_layer_fwd_fp16x2(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                             const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                             const float* W1, int F, const float* W2, const float* b2,
                             const float* W3, const float* b3, const float* w4, int update_coords, float* hn, float* x_out,
                             const float* h, int64_t ldh, const float* W5, const float* b5, const float* W6, const float* b6,
                             float* h_out, const float* W1n, const float* b1n, float* PQn, int next_kind,
                             int64_t n_nodes, int* status, void* stream);
/* operand-buffer depth of the warp-specialised edge forward kernel (csrc/egnn_tc2.cu): only 2 is accepted (a third
   buffer was measured without gain and no longer fits next to the padded operand tiles) */
int is_egnn_set_ws_buffers(int n);
/* variant bits of the warp-specialised edge forward kernel (A/B timing): bit 0 = A operand of MMA 2 from tensor memory
   (default on; results are bit-identical either way) */
int is_egnn_set_ws_variant(int bits);
/* node_mlp of layer l fused with the per-node half (P', Q') of layer l+1's first edge-MLP layer, on the
 * tensor cores (inference path).  W1n/b1n/PQn NULL = nothing follows.  next_kind 1: W1n = edge_mlp.0.weight
 * [64,130] of layer l+1, PQn [n,128].  next_kind 2 (after the last layer): W1n = [Wq;Wk;Wv] [192,64], b1n [192],
 * PQn = QKV [n,192], the projections of the per-graph attention (reference models/layers.py:13-16 / 67-69).
 * precision 0 = bf16, 3 = bf16x3, 4 = fp16x2 (inference forward). */
int is_egnn_node_post_pre_tc(const float* h, int64_t ldh, int F, const float* hn, const float* W5, const float* b5,
                             const float* W6, const float* b6, float* h_out, const float* W1n, const float* b1n,
                             float* PQn, int64_t n_nodes, int precision, int fast_act, int next_kind, void* stream);
int is_egnn_node_post_fwd(const float* h, int64_t ldh, int F, const float* hn, const float* W5, const float* b5,
                          const float* W6, const float* b6, float* h_out, int64_t n_nodes, void* stream);
/* gh_direct (the node_mlp's own gradient of h) and, in node_pre_bwd, gh (the gradient of the layer's input features) are
 * [n_nodes, F] row-major or NULL: F = 64 for a hidden layer, F = 20 for layer 0 (input gradients, attribution). */
int is_egnn_node_post_bwd(const float* gh_out, const float* h, int64_t ldh, int F, const float* hn,
                          const float* W5, const float* b5, const float* W6,
                          float* gh_direct, float* ghn, float* partials, int64_t n_nodes, void* stream);
/* tcgen05 (bf16x3, fp32-accurate) variant: same outputs, same partial layout, same grid. */
int is_egnn_node_post_bwd_tc(const float* gh_out, const float* h, int64_t ldh, int F, const float* hn,
                          const float* W5, const float* b5, const float* W6,
                          float* gh_direct, float* ghn, float* partials, int64_t n_nodes, void* stream);
int is_egnn_edge_bwd(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                     const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                     const float* W1, int F, const float* W2, const float* b2,
                     const float* W3, const float* b3, const float* w4,
                     const float* ghn, const float* gx_out,
                     float* gz1, float* gQ, float* gD, float* gxd, float* partials,
                     int64_t n_nodes, int* status, void* stream);
/* tcgen05 / TMEM variant of is_egnn_edge_bwd (bf16x3 operands, fp32-accurate; same outputs and partial layout) */
int is_egnn_edge_bwd_tc(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                        const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                        const float* W1, int F, const float* W2, const float* b2,
                        const float* W3, const float* b3, const float* w4,
                        const float* ghn, const float* gx_out,
                        float* gz1, float* gQ, float* gD, float* gxd, float* partials,
                        int64_t n_nodes, int* status, void* stream);
/* Two tile streams per CTA (csrc/egnn_bwd_ws.cu): same outputs and partial layout.  max_in_degree = DEVICE pointer
   to the batch's maximum in-degree (is_collate_csr's stats[0]): <= 112 runs the 112-edge-tile two-stream kernel,
   otherwise the lock-step kernel above (both are enqueued, the idle one returns at once); NULL = lock-step only. */
int is_egnn_edge_bwd_ws(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                        const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                        const float* W1, int F, const float* W2, const float* b2,
                        const float* W3, const float* b3, const float* w4,
                        const float* ghn, const float* gx_out,
                        float* gz1, float* gQ, float* gD, float* gxd, float* partials,
                        const int* max_in_degree, int64_t n_nodes, int* status, void* stream);
/* warps per tile stream of is_egnn_edge_bwd_ws: 8 (default), 12 or 16 (A/B timing; results identical up to the
   summation order of the bias-type gradients) */
int is_egnn_set_bwd_ws_warps(int n);
int is_egnn_node_pre_bwd(const float* gz1, const float* gQ, const float* gD, const float* gxd,
                         const float* gx_out, const float* gh_direct,
                         const int* outptr, const int* csc_pos, const float* h, int64_t ldh, int F,
                         const float* W1, float* gh, float* gx, float* partials, int64_t n_nodes, void* stream);
/* tcgen05 (bf16x3, fp32-accurate) variant: same outputs, same partial layout, same grid. */
int is_egnn_node_pre_bwd_tc(const float* gz1, const float* gQ, const float* gD, const float* gxd,
                         const float* gx_out, const float* gh_direct,
                         const int* outptr, const int* csc_pos, const float* h, int64_t ldh, int F,
                         const float* W1, float* gh, float* gx, float* partials, int64_t n_nodes, void* stream);
/* gradient of the scalar edge features: g_attr[csr_eid[p]] = (accumulate ? g_attr[csr_eid[p]] : 0) + sum_k gz1[p,k] *
 * W1[k, 2F+1] for every CSR position p.  gz1 [n_edges, 64] as written by the edge backward, g_attr [n_edges] in original
 * edge order; one launch per layer (accumulate = 0 for the first), deterministic (no atomics). */
int is_egnn_edge_attr_grad(const float* gz1, const int* csr_eid, const float* W1, int F, float* g_attr, int64_t n_edges,
                           int accumulate, void* stream);
int is_reduce_partials(const float* partials, int nparts, int64_t stride, float* out, void* stream);
/* the three partial buffers of one layer's backward (node_post, edge, node_pre) reduced by one launch */
int is_reduce_partials3(const float* p0, int n0, int64_t s0, float* o0, const float* p1, int n1, int64_t s1, float* o1,
                        const float* p2, int n2, int64_t s2, float* o2, void* stream);

/* ---- per-graph attention + global_mean_pool (models/layers.py:13-22,29-48,67-78;
 * models/hybrid_models.py:92-97 / 326-331).  QKV [n,192], O [n,64], LSE [n,H], pooled [B,64]. */
int is_attn_pool_fwd(const float* QKV, const int64_t* node_off, int n_graphs, int n_head, int max_nodes,
                     float* O, float* LSE, float* pooled, float* attn, const int64_t* attn_off, void* stream);
/* O == NULL (only with g_pooled != NULL and gO_full == NULL): the row statistics are recomputed and LSE [N, n_head] is
 * an output scratch -- for a forward pass that ran the pooled-rows-only kernel (is_attn_pool_infer_tc). */
int is_attn_pool_bwd(const float* QKV, const float* O, float* LSE, const int64_t* node_off, int n_graphs,
                     int n_head, int max_nodes, const float* g_pooled, const float* gO_full, float* gQKV, void* stream);
/* inference-only: pooled [B,64] from column sums of the attention matrix (no O / LSE / weights) */
int is_attn_pool_infer(const float* QKV, const int64_t* node_off, int n_graphs, int n_head, int max_nodes,
                       float* pooled, void* stream);

/* ---- fusion attention over the fused scalars + mean(dim=2) (models/hybrid_models.py:275,344-347;
 * comparative_models.py:392,484-486).  coef: [A(H) | C(H) | alpha(H) | beta(H) | btilde]. */
int is_fusion_attn_fwd(const float* c, int n_samples, int L, int n_head, const float* coef, float* out, void* stream);
int is_fusion_attn_bwd(const float* c, int n_samples, int L, int n_head, const float* coef, const float* gout,
                       float* gc, float* gcoef_part, void* stream);

/* ---- losses (utils/loss.py:13-31).  mode 0 = BCE-with-logits(pos_weight), 1 = MSE regression.
 * out: float[4] = {total, prediction, recon MSE, KLD}. */
int is_loss_fwd(const float* recon, const float* seq, int64_t n_recon, const float* mu, const float* logvar,
                int64_t n_lat, const float* logits, const float* y, int64_t B, int mode, float pos_weight,
                float w_pred, float w_mse, float w_kld, float* partial, float* out, void* stream);
int is_loss_bwd(const float* recon, const float* seq, int64_t n_recon, const float* mu, const float* logvar,
                int64_t n_lat, const float* logits, const float* y, int64_t B, int mode, float pos_weight,
                float w_pred, float w_mse, float w_kld, const float* gout,
                float* g_recon, float* g_mu, float* g_logvar, float* g_logits, void* stream);

/* ---- tcgen05 self-test: D[128,64] = A[128,64] * B[64,64]^T through the hand-written UMMA helpers
 * (csrc/umma.cuh).  mode 0 = bf16 operands, 1 = tf32, 2 = 3xTF32 split (fp32-accurate). */
/* Single-head per-graph attention + global mean pool on the tensor cores (inference: pooled rows only).  Same
 * result as is_attn_pool_infer with n_head = 1 (reference models/layers.py:13-22 / 67-78 + global_mean_pool,
 * hybrid_models.py:92-97 / 326-331).  QKV [N_total,192], node_off [n_graphs+1], pooled [n_graphs,64]; max_nodes <= 256;
 * precision 0 = bf16, 3 = bf16x3, 4 = fp16x2 (both fp32-accurate). */
int is_attn_pool_infer_tc(const float* QKV, const int64_t* node_off, int n_graphs, int max_nodes, int precision,
                          float* pooled, void* stream);
/* Backward of the pooled-rows-only single-head attention on the tensor cores (bf16x3, fp32-accurate;
 * csrc/attn_pool_bwd_tc.cu): what torch autograd derives for MultiHeadAttention + global_mean_pool in the reference
 * (models/layers.py:13-22 / 67-78, hybrid_models.py:92-97 / 326-331) when only the pooled rows feed the loss.  Same result
 * as is_attn_pool_bwd with n_head = 1, O = NULL, gO_full = NULL.  g_pooled [n_graphs,64] -> gQKV [N_total,192];
 * max_nodes <= 256. */
int is_attn_pool_bwd_tc(const float* QKV, const int64_t* node_off, int n_graphs, int max_nodes, const float* g_pooled,
                        float* gQKV, void* stream);
/* Compact input format -> dense model inputs, on the device and bit-exact (csrc/unpack.cu; SURVEY 8(f) row 1).
 * Replaces shipping the reference's fp32 one-hots over PCIe: x = [one_hot_20 | xyz] (data/utils.py:75-89,
 * preprocess.py:40-41,181), int64 endpoints, all-ones edge_attr (data/utils.py:60), [283,21] sequence one-hots. */
int is_unpack_nodes(const uint8_t* aa, const float* xyz, float* x, int64_t n_nodes, void* stream);
int is_unpack_edges(const int* src, const int* dst, const float* edge_attr, int64_t* src64, int64_t* dst64, float* attr_out,
                    int64_t n_edges, void* stream);
int is_onehot_tokens(const uint8_t* tokens, float* out, int64_t n_tokens, int vocab, void* stream);
/* Eval-mode small-layer fusions (csrc/head.cu; no autograd, dropout inactive).
 * is_vae_mid_infer: property_embedding (reference models/hybrid_models.py:46-52 / 280-286), mu / logvar = vae_fc21 /
 * vae_fc22 (h1), z = mu + eps exp(0.5 logvar) (:301-304, eps drawn by the caller), z_vae = [z | prop] (:339),
 * h3 = ReLU(vae_fc3 z_vae) (:306-307).  is_head_infer: x_gat = w_concat(pooled) (Wc NULL: identity), combined =
 * [x_gat | z_vae] (:341), closed-form fusion attention (coef NULL: none), classifier (:54-61, 351; W2 NULL: the 32
 * hidden features are returned). */
int is_vae_mid_infer(const float* h1, const float* prop, const float* eps, const float* Wp0, const float* bp0,
                     const float* Wp3, const float* bp3, const float* W21, const float* b21, const float* W22,
                     const float* b22, const float* W3, const float* b3, float* mu, float* logvar, float* z_vae,
                     float* h3, int n_samples, int hidden, int latent, int prop_dim, void* stream);
int is_head_infer(const float* pooled, const float* Wc, const float* bc, const float* z_vae, int LZ, const float* coef,
                  int n_head, const float* W1, const float* b1, const float* W2, const float* b2, int n_out,
                  float* x_gat, float* out, int n_samples, void* stream);
/* is_head_mc_infer: the head of is_head_infer (W2 [1,32] / b2 [1] required) for K reparameterisation draws of B samples.
 * Item i (n_items 1, or 2 for a cancer / wild-type pair) supplies pooled_i [B,64], mu_i / logvar_i [B,latent], z_vae_i
 * [B,latent+prop_dim] (only its property columns are read) and eps_i [K,B,latent]; z_i = mu_i + eps_i[k] exp(0.5
 * logvar_i) with the arithmetic of is_vae_mid_infer, tokens item-major [x_gat_0 | z_0 | prop_0 | x_gat_1 | ...] (at most
 * 256).  Draw k is bit-identical to is_head_infer on that draw.  -> logits [B,K], prob_mean / prob_std [B] (mean and
 * population standard deviation of sigmoid(logit) over the draws, fp64 accumulation in a fixed order, no atomics).
 * Item 1's pointers are ignored when n_items = 1. */
int is_head_mc_infer(const float* pooled0, const float* mu0, const float* logvar0, const float* z_vae0, const float* eps0,
                     const float* pooled1, const float* mu1, const float* logvar1, const float* z_vae1, const float* eps1,
                     int n_items, int latent, int prop_dim, const float* Wc, const float* bc, const float* coef, int n_head,
                     const float* W1, const float* b1, const float* W2, const float* b2, float* logits, float* prob_mean,
                     float* prob_std, int n_samples, int n_draws, void* stream);
/* is_head_features_infer: the classifier's hidden layer ReLU(W1 f + b1) [B,32] of the head of is_head_mc_infer at
 * z = mu (no noise), the features that the output layer reads (neighbors.embed).  Item i supplies pooled_i [B,64], mu_i
 * [B,latent] and z_vae_i [B,latent+prop_dim] (only its property columns are read); tokens item-major as in
 * is_head_mc_infer.  Bit-identical to the hid of is_head_infer on z_vae = [mu | prop].  Item 1's pointers are ignored
 * when n_items = 1. */
int is_head_features_infer(const float* pooled0, const float* mu0, const float* z_vae0, const float* pooled1,
                           const float* mu1, const float* z_vae1, int n_items, int latent, int prop_dim, const float* Wc,
                           const float* bc, const float* coef, int n_head, const float* W1, const float* b1, float* hid,
                           int n_samples, void* stream);
/* is_mutscan_expand (csrc/mutscan.cu): one pass of single-residue mutants for an in-silico saturation scan.  Copy k < r of
 * the base batch (x23 [N,23], node_off [B+1], seq [B,L,V]) carries sites[k] = (p, c) (int32 pairs): x23_out [r N, 23] and
 * seq_out [r B, L, V] are r copies of the base where, for every graph b with node_index[b,p] >= 0 (int64 [B,P], graph-local;
 * < 0 = absent site, copy unmodified), node row node_off[b] + node_index[b,p] of copy k has residue columns one_hot_20(c)
 * and sequence row seq_index[b,p] (int64 [B,P]) of sample b has one_hot_V(seq_columns[c]) (int64 [20]).  Bit-exact (copies
 * and 0.0 / 1.0 only).  flag (int32 [1], zeroed by the caller, never cleared) is set to 1 if a base site row is not exactly
 * one-hot, its sequence column is not seq_columns[its residue column], or an index is out of range (then that graph of
 * that copy is not patched).  No atomics, no synchronisation. */
int is_mutscan_expand(const float* x23, const int64_t* node_off, const int64_t* node_index, const float* seq,
                      const int64_t* seq_index, const int64_t* seq_columns, const int* sites, int r, int n_graphs, int n_sites,
                      int64_t n_nodes, int seq_len, int vocab, float* x23_out, float* seq_out, int* flag, void* stream);
/* is_variant_expand (csrc/mutscan.cu): one pass of a library of multi-site residue variants of a resident batch (x23
 * [N,23], node_off / edge_off [B+1], graph-local src_local / dst_local int64 [E], edge_attr [E,1], seq [B,L,V]).
 * Variant v < r is a copy of base graph b = sample[v] (int64 [r]): its x23 rows go to x23_out from row node_out[v], its
 * edges (endpoints still graph-local, attributes) to src_out / dst_out / edge_attr_out from edge_out[v] (node_out /
 * edge_out int64 [r+1]: the caller's running sums of the base counts), its sequence to seq_out[v] ([r,L,V]).  Then each
 * substitution s in offsets[v] .. offsets[v+1]-1 (int64 [r+1], indices into the n_subs-long int64 node_index /
 * seq_index / residue) writes one_hot_20(residue[s]) into the residue columns of node row node_index[s] (graph-local;
 * -1 = the graph does not hold that residue) and one_hot_V(seq_columns[residue[s]]) (int64 [20]) into sequence row
 * seq_index[s] (always required).  Bit-exact (copies and 0.0 / 1.0 only).  flag (int32 [1], zeroed by the caller, never
 * cleared) is set to 1, and the substitution is not applied, if a base row it replaces is not exactly one-hot (the x23
 * residue columns when node_index >= 0, the sequence row always), if both rows are present and the sequence's hot column
 * is not seq_columns[the row's residue column], or if an index is out of range; a sample outside [0, B) or output
 * offsets that disagree with the base counts or pass n_nodes_out / n_edges_out also raise it, and that variant is not
 * written.  Within one variant no row may be substituted twice (the last one in table order wins).  No atomics, no
 * synchronisation. */
int is_variant_expand(const float* x23, const int64_t* node_off, const int64_t* edge_off, const int64_t* src_local,
                      const int64_t* dst_local, const float* edge_attr, const float* seq, const int64_t* sample,
                      const int64_t* offsets, const int64_t* node_index, const int64_t* seq_index, const int64_t* residue,
                      const int64_t* seq_columns, const int64_t* node_out, const int64_t* edge_out, int r, int n_graphs,
                      int64_t n_subs, int seq_len, int vocab, int64_t n_nodes_out, int64_t n_edges_out, float* x23_out,
                      int64_t* src_out, int64_t* dst_out, float* edge_attr_out, float* seq_out, int* flag, void* stream);
/* is_design_expand / is_design_select (csrc/mutscan.cu): one round of a beam search over residue substitutions at the
 * n_sites = P <= 14 sites of is_mutscan_expand (node_index / seq_index int64 [B,P], -1 in both = absent site).  The beam
 * of sample b (beam = W <= 32 entries, of which the first n_states = Wt are read) is states int64 [B,W,P] (residue
 * columns, -1 at absent sites), keys int64 [B,W] (sum_p digit_p 20^p, digit 0 at absent sites), n_mut int64 [B,W]
 * (Hamming distance to native int64 [B,P]), valid uint8 [B,W]; allowed uint8 [B,P,20].  Slot k = (w P + p) 20 + c,
 * k < Wt P 20, is state w with site p set to residue c; it is valid when valid[b,w], site p is present, allowed[b,p,c],
 * c != states[b,w,p], the new state is within max_mutations of native, and no valid l < Wt equals the new state or,
 * with l < w, differs from it at exactly one site (an earlier slot yields it).
 * is_design_expand writes copies slot0 .. slot0 + r - 1 of the batch into x23_out [r N, 23] / seq_out [r B, L, V] (the
 * layout of is_mutscan_expand): every present site of graph b gets the residue of state w, site p gets c if the slot is
 * valid for b (an invalid slot is written as its parent state).  Bit-exact (copies and 0.0 / 1.0 only).  flag (int32 [1],
 * zeroed by the caller, never cleared) is set to 1 if the base rows of site p are not exactly one-hot or contradict
 * seq_columns, or an index or residue is out of range (that site is not written).
 * is_design_select, one CTA per sample: the pool is the Wt carried entries (with logits [B,W,K], prob_mean / prob_std
 * [B,W]) and the valid slots (round_logits [Wt P 20, B, K], round_mean / round_std [Wt P 20, B]); an entry's objective is
 * fmaf(kappa, prob_std, prob_mean) in fp32, and entries whose objective is NaN (or that are invalid) are never taken.  The
 * next beam (the *_out buffers, same shapes, must not alias the inputs) is the top W of the pool by objective
 * (descending when maximize != 0, else ascending), ties to the smaller key; entries past the pool's size are invalid and
 * hold the native state with NaN scores.  best[b * best_stride] = the objective of entry 0 (NaN if none).
 * Deterministic, no atomics. */
int is_design_expand(const float* x23, const int64_t* node_off, const int64_t* node_index, const float* seq,
                     const int64_t* seq_index, const int64_t* seq_columns, const int64_t* states, const int64_t* n_mut,
                     const unsigned char* valid, const int64_t* native, const unsigned char* allowed, int slot0, int r, int n_graphs, int n_sites, int beam, int n_states, int max_mutations, int64_t n_nodes,
                     int seq_len, int vocab, float* x23_out, float* seq_out, int* flag, void* stream);
int is_design_select(const int64_t* states, const int64_t* keys, const int64_t* n_mut, const unsigned char* valid,
                     const float* logits, const float* prob_mean, const float* prob_std, const float* round_logits,
                     const float* round_mean, const float* round_std, const int64_t* native, const unsigned char* allowed,
                     const int64_t* node_index, int n_graphs, int n_sites, int beam, int n_states, int n_draws,
                     int max_mutations, float kappa, int maximize, int64_t* states_out, int64_t* keys_out,
                     int64_t* n_mut_out, unsigned char* valid_out, float* logits_out, float* mean_out, float* std_out,
                     float* objective_out, float* best, int64_t best_stride, void* stream);
/* is_occlusion_expand (csrc/occlusion.cu): one pass of single-removal structural variants of a resident batch (x23
 * [N,23], node_off / edge_off [B+1], graph-local src_local / dst_local int64 [E], edge_attr [E,1]).  Variant v < r is a
 * copy of base graph b = sample[v] (int64 [r]) with one removal: node_b[v] == -1 occludes graph-local row a = node_a[v]
 * (its 23 floats become 0.0 and every edge with src == a or dst == a is dropped), node_b[v] >= 0 occludes the contact
 * {a, node_b[v]} (every edge a -> node_b or node_b -> a is dropped; rows unchanged, self-loops never dropped).  Its x23
 * rows go to x23_out from row node_out[v], its kept edges, in base order, with graph-local endpoints and their
 * attributes, to src_out / dst_out / edge_attr_out from edge_out[v] (node_out / edge_out int64 [r+1]: the caller's
 * running sums of the node counts and of the kept edge counts).  Bit-exact (copies and 0.0 only).  flag (int32 [1],
 * zeroed by the caller, never cleared) is set to 1, and that variant is not written, for a sample outside [0, B), node_a
 * outside [0, n_b), node_b outside [-1, n_b) or equal to node_a, node_out[v+1] - node_out[v] != n_b, a kept count that
 * is not edge_out[v+1] - edge_out[v], or offsets past n_nodes_out / n_edges_out.  No atomics. */
int is_occlusion_expand(const float* x23, const int64_t* node_off, const int64_t* edge_off, const int64_t* src_local,
                        const int64_t* dst_local, const float* edge_attr, const int64_t* sample, const int64_t* node_a,
                        const int64_t* node_b, const int64_t* node_out, const int64_t* edge_out, int r, int n_graphs,
                        int64_t n_nodes_out, int64_t n_edges_out, float* x23_out, int64_t* src_out, int64_t* dst_out,
                        float* edge_attr_out, int* flag, void* stream);
/* is_coord_noise_expand (csrc/coordnoise.cu): one pass of r seeded coordinate perturbations of a resident batch (x23
 * [N,23], node_off [B+1], sigma fp32 [N] per node row), in the layout of GraphBatch.replicate(r): x23_out [r N, 23],
 * copy k of graph b at rows k N + node_off[b].  Copy k is structure draw m = draw0 + k: graph-local row a of graph b
 * keeps columns 0..19 and gets x_c + sigma z_c (fmaf) in columns 20..22, z = three standard normals of Philox4x32-10
 * with counter (a, b, m, item) and key (low, high 32 bits of seed), by Box-Muller on u_j = ((v_j >> 8) + 0.5) 2^-24:
 * z0 = sqrt(-2 log u0) cospi(2 u1), z1 = sqrt(-2 log u0) sinpi(2 u1), z2 = sqrt(-2 log u2) cospi(2 u3).  Rows with
 * sigma == 0 are copied bit-exact.  No device flag: the caller checks every argument (draw0 + r <= 2^32).  No atomics. */
int is_coord_noise_expand(const float* x23, const int64_t* node_off, const float* sigma, int r, int n_graphs,
                          int64_t n_nodes, uint64_t seed, uint32_t item, uint32_t draw0, float* x23_out, void* stream);
/* Shapley values over structural removals (csrc/shapley.cu).  players int32 [N]: the graph-local player id of each node
 * row, -1 for a row never removed; sample b has P_b = player_off[b+1] - player_off[b] <= 256 players (ids 0 .. P_b - 1)
 * and var_off[b+1] - var_off[b] = 1 + T (P_b - 1) variants (0 without players): the empty coalition (every player
 * removed) first, then coalitions j = 1 .. P_b - 1 of permutation t = 0 .. T-1, t ascending then j ascending.  Removing
 * a player zeroes the 23 floats of its rows and drops every edge touching one of them; kept edges keep their base order.
 * The flag (int32 [1], zeroed by the caller, never cleared) is set to 1 for tables that disagree with the batch.
 *
 * is_shapley_plan: T even in [2, 2^16].  ranks int32 [B, T, max_players]: row 2u of sample b ranks its players by the
 * key v0 of Philox4x32-10 with counter (p, b, u, 2) and key (low, high 32 bits of seed), ties to the smaller id; row
 * 2u+1 is P_b - 1 minus row 2u; entries past P_b are -1.  kept int64 [V]: the kept-edge count of every variant.  Flag:
 * P_b > min(256, max_players) or a variant count that is not 1 + T (P_b - 1).  Integer counts, no float atomics. */
int is_shapley_plan(const int64_t* node_off, const int64_t* edge_off, const int64_t* src_local, const int64_t* dst_local,
                    const int* players, const int64_t* player_off, const int64_t* var_off, int n_graphs,
                    int permutations, int max_players, uint64_t seed, int* ranks, int64_t* kept, int* flag,
                    void* stream);
/* is_shapley_expand: one pass of r coalition variants of a resident batch (inputs as is_occlusion_expand).  Variant v is
 * base graph b = sample[v] with every row i removed for which players[i] >= 0 and ranks[rank_row[v]][players[i]] <
 * threshold[v] (ranks int32 [n_rank_rows, max_players]); its rows go to x23_out from row node_out[v], its kept edges to
 * src_out / dst_out / edge_attr_out from edge_out[v].  Bit-exact (copies and 0.0 only).  Flag, and that variant not
 * written: sample outside [0, B), rank_row outside [0, n_rank_rows), threshold outside [0, max_players], n_b > 256, a
 * player id >= max_players, node_out[v+1] - node_out[v] != n_b, a kept count that is not edge_out[v+1] - edge_out[v], or
 * offsets past n_nodes_out / n_edges_out.  No atomics. */
int is_shapley_expand(const float* x23, const int64_t* node_off, const int64_t* edge_off, const int64_t* src_local,
                      const int64_t* dst_local, const float* edge_attr, const int* players, const int* ranks,
                      const int64_t* sample, const int64_t* rank_row, const int64_t* threshold, const int64_t* node_out,
                      const int64_t* edge_out, int r, int n_graphs, int64_t n_rank_rows, int max_players,
                      int64_t n_nodes_out, int64_t n_edges_out, float* x23_out, int64_t* src_out, int64_t* dst_out,
                      float* edge_attr_out, int* flag, void* stream);
/* Shapley values of contacts and contact groups (csrc/shapley.cu): the players are sets of edges.  edge_players int32
 * [E]: the graph-local player id of each edge, -1 for an edge never removed.  Removing a player drops its edges; rows,
 * the attributes of the kept edges and their base order are unchanged.  Tables, variant order and flag as above.
 *
 * is_shapley_edge_plan: as is_shapley_plan, the keys with counter (p, b, u, 3).  An edge of player q is kept in
 * coalition j of permutation t iff j <= rank_t(q); an edge with id -1 (or outside [0, P_b)) always.  max_players <= 256.
 * edge_players may be NULL when the batch has no edge. */
int is_shapley_edge_plan(const int64_t* edge_off, const int* edge_players, const int64_t* player_off,
                         const int64_t* var_off, int n_graphs, int permutations, int max_players, uint64_t seed,
                         int* ranks, int64_t* kept, int* flag, void* stream);
/* is_shapley_edge_expand: as is_shapley_expand, with every row copied verbatim and every edge e with edge_players[e] >= 0
 * and ranks[rank_row[v]][edge_players[e]] < threshold[v] dropped.  Flag, and that variant not written: sample outside
 * [0, B), rank_row outside [0, n_rank_rows), threshold outside [0, max_players], an edge player id >= max_players,
 * node_out[v+1] - node_out[v] != n_b, a kept count that is not edge_out[v+1] - edge_out[v], or offsets past n_nodes_out /
 * n_edges_out.  Bit-exact (copies only), no atomics. */
int is_shapley_edge_expand(const float* x23, const int64_t* node_off, const int64_t* edge_off,
                           const int64_t* src_local, const int64_t* dst_local, const float* edge_attr,
                           const int* edge_players, const int* ranks, const int64_t* sample, const int64_t* rank_row,
                           const int64_t* threshold, const int64_t* node_out, const int64_t* edge_out, int r,
                           int n_graphs, int64_t n_rank_rows, int max_players, int64_t n_nodes_out,
                           int64_t n_edges_out, float* x23_out, int64_t* src_out, int64_t* dst_out,
                           float* edge_attr_out, int* flag, void* stream);
/* is_shapley_reduce: logits [V, K] of the variants, base_logits [B, K] of the unmodified batch, ranks [B, T,
 * max_players] as is_shapley_plan writes them.  v_logit = mean over k of the logit, v_prob = mean of sigmoid(logit), in
 * fp64; the player at position j-1 of permutation t gets Δ = v(t, j-1) - v(t, j) (j = 0: base, j = P_b: the empty
 * variant); d_u = (Δ_2u + Δ_2u+1) / 2; phi = mean over u of d_u and se = sqrt(Σ_u (d_u - phi)^2 / (U (U - 1))), U = T/2
 * (NaN for U = 1), accumulated over u ascending, rounded to fp32 into phi_* / se_* [Q] at player_off[b] + p.
 * gap_* [B] = (v(base) - v(empty)) - Σ_p phi(p) (0 without players).  Flag: the variant tables or a rank outside
 * [0, P_b).  Deterministic, no atomics. */
int is_shapley_reduce(const float* logits, const float* base_logits, const int* ranks, const int64_t* player_off,
                      const int64_t* var_off, int n_graphs, int permutations, int max_players, int n_draws,
                      int64_t n_variants, float* phi_logit, float* phi_prob, float* se_logit, float* se_prob,
                      float* gap_logit, float* gap_prob, int* flag, void* stream);
/* Dense Linear layer on the tensor cores: C[M,N] = act(A[M,K] W[N,K]^T + bias), fp32 in / out, operands split
 * on the fly into three bf16 terms (precision 3, fp32-accurate) or rounded to bf16 (precision 0).  Replaces the
 * nn.Linear layers of the sequence VAE (reference models/hybrid_models.py:63-74: vae_fc1 with ReLU, vae_fc4) in the
 * no-grad path.  lda / ldw / ldc = row strides in floats (any alignment); bias may be NULL; split_k > 1 (see
 * is_linear_tc_split_k) needs workspace >= split_k * M * N floats and sums the K slices in order (deterministic). */
int is_linear_tc_split_k(int64_t M, int64_t N, int64_t K);
int is_linear_tc(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, float* C, int64_t ldc,
                 int64_t M, int64_t N, int64_t K, int relu, int precision, int split_k, float* workspace, void* stream);
int is_umma_selftest(const float* A, const float* B, float* D, int mode, void* stream);
/* cycles per tcgen05.mma (96 MMAs of N = 64, bf16, issue to completion) for 16 operand-layout / accumulator-rotation
   configurations of the edge kernels (csrc/umma_selftest.cu: umma_timing_kernel; scripts/umma_timing.py): out[16] */
int is_umma_timing(float* out, void* stream);

/* ---- TMA-fed tcgen05 GEMM for the dense Linear layers, forward and backward (csrc/gemm_tma.cu): the nn.Linear
 * layers of the sequence VAE (models/hybrid_models.py:63-74 / 297-308) and what autograd derives for them.
 * is_split_planes: fp32 X [R, C] (row stride ld) -> bf16 planes (a = a1 + a2 + a3; n_planes 3, or 1 = rounded) in
 *   row-major [n_planes][R][Cp] and / or transposed [n_planes][C][Rp] form (Cp / Rp = C / R rounded up to 8, zero
 *   padded); optional ReLU mask (X kept where relu_src > 0), per-row-block column sums colsum_part [gr][C] with
 *   gr = ceil((planes_t ? Rp : R) / 32) (bias gradient: sum with is_reduce_partials), resid_flag set to 1 if X is
 *   not exact in bf16 (caller zeroes it first).
 * is_gemm_planes_tma: C[M, N] = act(A B^T + bias) from planes A [n_planes][M][Kp], B [n_planes][N][Kp]; operand tiles
 *   arrive by cp.async.bulk.tensor (128-byte swizzle), six bf16 partial products accumulate in TMEM (fp32-accurate);
 *   a/b_resid_flag (device, or NULL) = 0 skips the products of that operand's second / third plane.  split_k > 1
 *   (is_gemm_tma_split_k) needs workspace >= split_k * M * N floats; slices are summed in order (deterministic). */
int is_gemm_tma_split_k(int64_t M, int64_t N, int64_t Kp);
int is_split_planes(const float* X, int64_t ld, int64_t R, int64_t C, const float* relu_src, int64_t ld_relu, int n_planes,
                    void* planes, void* planes_t, float* colsum_part, int* resid_flag, void* stream);
int is_gemm_planes_tma(const void* A_planes, int64_t M, const void* B_planes, int64_t N, int64_t Kp, int n_planes,
                       const int* a_resid_flag, const int* b_resid_flag, const float* bias, int relu, float* C, int64_t ldc,
                       int split_k, float* workspace, void* stream);

/* ---- segment pooling (csrc/segment_pool.cu): torch_geometric.nn.global_mean_pool / global_max_pool
 * (models/hybrid_models.py:97,331; models/ablation_models.py:296-297).  X [n, C] with row stride ldx, segments =
 * node_off [n_graphs + 1]; mode 0 mean, 1 max (0 for an empty segment), 2 sum; out [n_graphs, C].  Backward of max
 * splits the gradient evenly among the rows attaining the maximum (scatter_reduce 'amax'); `pooled` = forward output. */
int is_segment_pool_fwd(const float* X, int64_t ldx, int C, const int64_t* node_off, int n_graphs, int mode,
                        float* out, void* stream);
int is_segment_pool_bwd(const float* X, int64_t ldx, int C, const int64_t* node_off, int n_graphs, int mode,
                        const float* pooled, const float* g_out, float* gX, int64_t ldg, void* stream);

/* ---- PairedContrastiveLoss (utils/contrastive.py:37-83; csrc/contrastive.cu): projector Linear(D, Z, no bias) ->
 * BatchNorm1d (batch statistics; running statistics updated for the cancer then the wild-type call when the gate is
 * open) -> ReLU -> Linear(Z, Z, no bias); centring, std hinge, pair-similarity and cross-correlation terms; the
 * "exactly two target values" gate is evaluated on the device.  out [4] = {loss, pair, corr, std}.  scratch:
 * is_contrastive_scratch_floats(B, Z) floats written by the forward and read by the backward; work: 4 * B * Z floats.
 * Parameter-gradient outputs of the backward may be NULL. */
int64_t is_contrastive_scratch_floats(int B, int Z);
int is_contrastive_fwd(const float* Ec, const float* Ew, const float* target, int B, int D, int Z, const float* W1,
                       const float* gamma, const float* beta, const float* W2, float bn_eps, float momentum,
                       float* run_mean, float* run_var, int64_t* n_tracked, float lambda_off, float* scratch, float* out,
                       void* stream);
int is_contrastive_bwd(const float* Ec, const float* Ew, int B, int D, int Z, const float* W1, const float* gamma,
                       const float* beta, const float* W2, const float* scratch, const float* gout, float* work,
                       float* gEc, float* gEw, float* gW1, float* g_gamma, float* g_beta, float* gW2, void* stream);

/* ---- fused Adam / AdamW step over a flat fp32 buffer (csrc/optim.cu): torch.optim.Adam / AdamW as constructed at
 * train_IEDB_wFT.py:74,97 and train_Cancer_wFT.py:98,122, stepped at procedures/train.py:28,122.  decoupled = 1 is
 * AdamW.  step_size = lr / (1 - beta1^t), inv_bc2_sqrt = 1 / sqrt(1 - beta2^t); grad_scale multiplies g first. */
int is_fused_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int decoupled, float step_size, float inv_bc2_sqrt, float grad_scale, void* stream);

/* capturable form: the step count is a device float (`tick` != 0 increments it first), bias corrections on the device */
int is_fused_adam_capturable(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                             float eps, float weight_decay, int decoupled, float* step, int tick, float grad_scale,
                             void* stream);

/* ---- on-device training augmentations (csrc/augment.cu; SURVEY 8(f) row 2) ------------------------------------
 * is_rotate_coords: RandomRotation (data/utils.py:148-155): x[:, c0:c0+3] @= Q_g, Q_g = Householder-QR orthogonal factor
 *   (LAPACK sign convention = numpy.linalg.qr) of the caller's 3x3 normal draw M_g; Qout [n_graphs, 9] or NULL.
 * is_mask_single_residue: mask_single_structure (data/immmunopred_dataloader.py:104-115, :248-266): residue
 *   floor(u_g * n_valid) of graph g's valid residues (optionally of type want_aa[g]) gets an all-ones one-hot;
 *   aa_out = its type (0 if none), node_out = its row (-1 if none) or NULL.
 * is_mask_rows: mask_structure (:92-102; fill_col < 0: zero the one-hot unless the row sums to more than 1) and
 *   mask_sequence (:78-90; fill_col = padding token): the `count` smallest keys among the first limit[g] rows
 *   (limit NULL: all) of every segment. */
int is_rotate_coords(float* x, int64_t ldx, int c0, const int64_t* node_off, int n_graphs, const float* M, float* Qout,
                     void* stream);
int is_mask_single_residue(float* x, int64_t ldx, int n_feat, const int64_t* node_off, int n_graphs, const float* u,
                           const int64_t* want_aa, int64_t* aa_out, int64_t* node_out, void* stream);
int is_mask_rows(float* data, int64_t ld, int n_cols, const int64_t* seg_off, const int64_t* limit, int n_segments,
                 const float* keys, int count, int fill_col, int max_rows, void* stream);

/* ---- exact k-nearest-neighbour search (csrc/knn.cu; neighbors.nearest) ---------------------------------------------
 * query [Q, D], bank [R, D] fp32 row-major; 1 <= k <= 64, 1 <= D <= 256, 1 <= R < 2^31; exclude int64 [Q] (the bank row
 * query q must not return, -1 = none; every entry in [-1, R)) or NULL.
 *   distance: squared Euclidean in fp32, one rounding sequence per pair: acc = 0; for d = 0 .. D-1 ascending, t = q_d -
 *     r_d, acc = fmaf(t, t, acc); independent of tiling, slicing and Q.  One metric: pass L2-normalised rows for cosine
 *     order (|a - b|^2 = 2 - 2 cos).
 *   order: ascending in (distance, bank index), ties to the smaller index; bit-identical for any slice count.
 *   missing data: a pair whose distance is NaN is never returned (a bank row or a query with a NaN feature); unfilled
 *     slots hold index -1 and distance +inf.
 * slices S in [1, min(65535, ceil(R / 128))]: the bank is split among S CTAs per query tile; S > 1 needs workspace
 * uint64 [Q, S, k] and adds one merge kernel.  -> index int64 [Q, k], distance fp32 [Q, k]. */
int is_knn(const float* query, const float* bank, const int64_t* exclude, int64_t n_query, int64_t n_bank, int dim, int k,
           int slices, unsigned long long* workspace, int64_t* index, float* distance, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IMMUNOSTRUCT_B200_H */
