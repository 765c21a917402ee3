/*
 * step_b200.h - C ABI of the B200-native STEP hot path (libstep_b200.so).
 *
 * The reference (GestaltCogTeam/STEP) is pure Python/PyTorch and has no native
 * interface; every entry point below replaces a span of reference Python that
 * PyTorch-eager executes as a chain of library kernels.  The span is cited as
 * file:line relative to the reference repository root.
 *
 * Conventions (SURVEY.md section 8(b)):
 *   - plain `extern "C"`, pointers + sizes only, no torch / C++ types;
 *   - every pointer is a DEVICE pointer unless its name starts with `h_`;
 *   - the caller allocates every input, output and workspace buffer; the
 *     callee never allocates, frees or retains a pointer past return;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*), the call
 *     returns without synchronising;
 *   - return value: 0 ok, <0 bad argument / unsupported shape (see
 *     step_last_error_string), >0 a cudaError_t from the launch;
 *   - all floating point buffers are fp32, row-major, densely packed unless a
 *     stride argument says otherwise.
 */
#ifndef STEP_B200_H_
#define STEP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STEP_B200_ABI_VERSION 3

#define STEP_OK 0
#define STEP_EINVAL (-1)
#define STEP_EUNSUPPORTED (-2)
#define STEP_EWORKSPACE (-3)

int step_abi_version(void);
/* The library carries its own (statically linked) CUDA runtime; select the device the following
 * calls of this host thread launch on (the caller's framework keeps a separate "current device"). */
int step_set_device(int device);
/* Text of the last error raised on the calling thread ("" if none). */
const char *step_last_error_string(void);

/* Number of CUDA kernels this library has enqueued since it was loaded (all streams / devices; memsets are not
 * kernels and are not counted).  bench.py reports the difference across its timed region as `gpu_launches`. */
unsigned long long step_launch_count(void);

/* ------------------------------------------------------------------------ *
 * TSFormer encoder, forecasting mode (frozen, forward only)
 *   step/step_arch/tsformer/tsformer.py:86-105,189-191
 * ------------------------------------------------------------------------ */

/* One nn.TransformerEncoderLayer(96, 4, 384) worth of weights
 * (step/step_arch/tsformer/transformer_layers.py:10-11; state-dict names in
 * SURVEY.md Appx C). */
typedef struct step_ts_layer_weights {
  const float *in_proj_w;  /* [288, 96] */
  const float *in_proj_b;  /* [288]     */
  const float *out_proj_w; /* [96, 96]  */
  const float *out_proj_b; /* [96]      */
  const float *lin1_w;     /* [384, 96] */
  const float *lin1_b;     /* [384]     */
  const float *lin2_w;     /* [96, 384] */
  const float *lin2_b;     /* [96]      */
  const float *norm1_w, *norm1_b, *norm2_w, *norm2_b; /* [96] each */
} step_ts_layer_weights;

/* Patch embedding + positional embedding + sqrt(d) scaling:
 *   patch.py:31-42 (Conv2d(1,96,(12,1),stride 12) == [12]->[96] map per patch),
 *   positional_encoding.py:24-35, transformer_layers.py:15.
 * series element (b, t, n) is read at series[b*sB + t*sT + n*sN] (element
 * strides, so a channel-0 view of long_history [B, P*12, N, C] needs no copy).
 * x: [B*N*P, 96], token order (b, n, p).
 * drop_p > 0 applies inverted dropout with the counter-based generator keyed
 * by `seed` (reference: positional_encoding.py:32 while the module is in
 * train()); drop_p == 0 is the deterministic parity path. */
int step_ts_embed_fwd(const float *series, long long sB, long long sT, long long sN, int B, int N, int P,
                      const float *patch_w /*[96,12]*/, const float *patch_b /*[96]*/,
                      const float *pos /*[>=P,96]*/, float *x, float drop_p, unsigned long long seed,
                      void *stream);

/* C[M,Nout] = A[M,K] * W[Nout,K]^T + bias, then
 *   epilogue 0: nothing, 1: ReLU,
 *   epilogue 2 (Nout == 96 only): C = LayerNorm(residual + drop(C)) * ln_w + ln_b, eps 1e-5
 *     (the post-norm residual blocks of nn.TransformerEncoderLayer).
 * drop_p / seed / drop_site: inverted dropout on the GEMM result (before the residual add /
 * after the ReLU), 0 disables. */
int step_linear_f32(const float *A, const float *W, const float *bias, float *C, long long M, int K, int Nout,
                    int epilogue, const float *residual, const float *ln_w, const float *ln_b,
                    float drop_p, unsigned long long seed, unsigned drop_site, void *stream);

/* Multi-head self attention over S independent sequences of P tokens, 4 heads x 24:
 *   softmax(q k^T / sqrt(24)) v   (torch MultiheadAttention as used at
 *   transformer_layers.py:10-18, no mask).  qkv: [S*P, 288] = (q | k | v),
 * heads are contiguous 24-wide slices; out: [S*P, 96].  drop_p: dropout on the
 * attention probabilities. */
int step_attn_fwd_f32(const float *qkv, float *out, int S, int P, float drop_p, unsigned long long seed,
                      unsigned drop_site, void *stream);

/* Row LayerNorm over 96 features (encoder_norm, tsformer.py:103). */
int step_layernorm96_f32(const float *x, const float *w, const float *b, float *y, long long M, void *stream);

/* Bytes of workspace step_ts_encoder_fwd needs for `chunk_seqs` sequences of P tokens in flight. */
size_t step_ts_encoder_workspace_bytes(int chunk_seqs, int P);

/* Whole frozen encoder: series -> hidden [B, N, P, 96] (tsformer.py:189-191).
 * Sequences are processed `chunk_seqs` at a time so that the per-layer
 * intermediates of a chunk stay L2-resident (chunk_seqs <= 0: all at once).
 * drop_p: dropout probability of every dropout site inside TSFormer (the
 * reference leaves the frozen TSFormer in train() during STEP training). */
int step_ts_encoder_fwd(const float *series, long long sB, long long sT, long long sN, int B, int N, int P,
                        const float *patch_w, const float *patch_b, const float *pos,
                        const step_ts_layer_weights *h_layers, int n_layers,
                        const float *final_norm_w, const float *final_norm_b, float *hidden,
                        void *workspace, size_t workspace_bytes, int chunk_seqs,
                        float drop_p, unsigned long long seed, void *stream);

/* The transformer layer stack alone, on caller-provided tokens x [S*P, 96] (already multiplied by sqrt(96));
 * x is replaced by the output, fnw/fnb (both or neither) = a final LayerNorm fused into the last epilogue.
 * Used by TSFormer(mode="pre-train") for the encoder over the unmasked tokens and for the decoder
 * (reference tsformer.py:86-136, transformer_layers.py:13-20).  workspace: step_ts_encoder_workspace_bytes(S, P). */
int step_ts_layers_fwd(float *x, int S, int P, const step_ts_layer_weights *L, int n_layers, const float *fnw,
                       const float *fnb, void *workspace, size_t workspace_bytes, float drop_p,
                       unsigned long long seed, void *stream);


/* ------------------------------------------------------------------------ *
 * TSFormer pre-training (stage 1): backward building blocks of the masked auto-encoder
 *   step/step_arch/tsformer/tsformer.py:71-160, transformer_layers.py:10-20 (the reference differentiates through autograd)
 * ------------------------------------------------------------------------ */
/* Backward of step_attn_fwd_f32: dqkv [S*P, 288] from dout [S*P, 96]; out = the forward's output; the dropout mask is
 * regenerated from (seed, drop_site).  scratch: S*4*P*2 floats. */
int step_attn_bwd_f32(const float *qkv, const float *out, const float *dout, int S, int P, float drop_p, unsigned long long seed,
                      unsigned drop_site, float *scratch, float *dqkv, void *stream);
/* y = LayerNorm96(x + r) * w + b (r may be NULL); sum [M,96] = x + r and stat [M,2] = (mean, rstd) are kept for backward
 * (either may be NULL for inference). */
int step_add_layernorm96_fwd(const float *x, const float *r, const float *w, const float *b, long long M, float *sum, float *stat,
                             float *y, void *stream);
/* dx [M,96] (the gradient of both x and r), dw [96], db [96]. */
int step_add_layernorm96_bwd(const float *dy, const float *sum, const float *stat, const float *w, long long M, float *dx,
                             float *dw, float *db, void *stream);
/* Inverted dropout with the counter-based generator: y = x * keep / (1 - p); calling it on dy with the same
 * (seed, site) is the backward.  n must be a multiple of 4. */
int step_dropout_f32(const float *x, long long n, float drop_p, unsigned long long seed, unsigned site, float *y, void *stream);

/* ------------------------------------------------------------------------ *
 * TSFormer encoder, bf16 tensor-core path (tcgen05.mma + TMEM + TMA bulk copies)
 * Same reference spans as the fp32 path above.  Activations travel between kernels as
 * "tile images": a [T, K] bf16 matrix stored as [T/128][K/8][128 rows][8] (the UMMA K-major
 * no-swizzle canonical layout of a 128-row tile), weights as [K/8][Nout][8].
 * ------------------------------------------------------------------------ */
typedef struct step_ts_layer_images {
  const void *in_proj;  /* [12][288][8] bf16 */
  const void *out_proj; /* [12][96][8]  */
  const void *lin1;     /* [12][384][8] */
  const void *lin2;     /* [48][96][8]  */
  /* Optional (NULL = run the four token GEMMs as separate launches): the weights of the fused token-block kernel as
   * twelve [12][96][8] slices (18432 B each) in program order: out_proj | lin1 rows 0-95, lin2 K-columns 0-95, ... (x4) |
   * the NEXT layer's in_proj rows 0-95 (q), 96-191 (k), 192-287 (v); the last layer carries the first nine only. */
  const void *fused;
} step_ts_layer_images;

/* fp32 W [Nout][K] -> bf16 weight image [K/8][Nout][8] (Nout*K*2 bytes). */
int step_tc_pack_weight(const float *w, int Nout, int K, void *img, void *stream);
/* row-major fp32 [T][K] <-> activation tile image (ceil(T/128)*K*256 bytes); test / debug helpers. */
int step_tc_rows_to_image(const float *x, long long T, int K, void *img, void *stream);
int step_tc_image_to_rows(const void *img, long long T, int K, float *x, void *stream);
/* out = epilogue(A W^T + bias) on tcgen05.  K in {96, 384}, Nout in {96, 192, 288, 384}.
 *   mode 0: out_f32 [T][Nout] row-major;  mode 1: ReLU -> out_img (K' = Nout);
 *   mode 2 (Nout == 96): LayerNorm(residual image + .) -> out_img and/or out_f32 [T][96]. */
int step_tc_linear(const void *a_img, const void *w_img, const float *bias, long long T, int K, int Nout, int mode,
                   const void *res_img, const float *ln_w, const float *ln_b, void *out_img, float *out_f32, void *stream);
/* Patch + positional embedding (x sqrt(96), positional dropout) straight into the X tile image [B*N*P, 96] - the first
 * kernel of step_ts_encoder_fwd_bf16, exposed for the per-site dropout tests. */
int step_tc_embed_fwd(const float *series, long long sB, long long sT, long long sN, int B, int N, int P, const float *patch_w,
                      const float *patch_b, const float *pos, void *x_img, float drop_p, unsigned long long seed, void *stream);
/* Same as step_tc_linear for modes 1 and 2 with the dropout site of that epilogue live (inverted dropout on the ReLU
 * output / on the GEMM result before the residual add; transformer_layers.py:10-11 -> nn.TransformerEncoderLayer's
 * dropout, dropout1, dropout2), drawn from the counter-based generator keyed by `seed`. */
int step_tc_linear_drop(const void *a_img, const void *w_img, const float *bias, long long T, int K, int Nout, int mode,
                        const void *res_img, const float *ln_w, const float *ln_b, void *out_img, float *out_f32,
                        float drop_p, unsigned long long seed, void *stream);
/* Bytes of the per-(sequence, head) attention operand images: which = 0 -> Q, 1 -> K (== V), 2 -> the row-maximum bound
 * workspace (S*4 floats max_j |k_j| followed by S*4*P floats |q_i|). */
size_t step_tc_attn_image_bytes(int S, int P, int which);
/* QKV projection of an X image [S*P, 96] straight into the attention operand images (Q pre-scaled by
 * log2(e)/sqrt(24); the last row tile of odd heads is placed at tile rows 64.. when it holds <= 64 queries).
 * `bound` (may be NULL): workspace of step_tc_attn_image_bytes(S, P, 2) bytes that receives the operand norms. */
int step_tc_qkv(const void *x_img, const void *w_img, const float *bias, int S, int P, void *q_img, void *k_img, void *v_img,
                float *bound, void *stream);
/* softmax(Q K^T) V per (sequence, head) on tcgen05 -> O tile image [S*P, 96]
 * (transformer_layers.py:13-20 -> nn.MultiheadAttention inside nn.TransformerEncoderLayer).  P <= 352
 * (P > 176 runs the key-split variant: two 176-key blocks per row tile merged in shared memory).
 * `bound` (may be NULL): the workspace step_tc_qkv filled; rows whose Cauchy-Schwarz bound |q_i| max_j |k_j| is <= 40
 * (log2 domain) are exponentiated in one pass against that bound, all others (and every row when NULL) take the exact
 * two-pass row maximum.  Both are the same softmax up to bf16 rounding of the probabilities. */
int step_tc_attention(const void *q_img, const void *k_img, const void *v_img, void *o_img, const float *bound, int S, int P,
                      float drop_p, unsigned long long seed, void *stream);
/* Host-only arithmetic: the bf16x2 threshold of the attention-probability dropout (transformer_layers.py:10-11 -> the dropout
 * inside nn.MultiheadAttention).  A probability is kept iff the 16-bit half of its random word, read as a bf16 number, is
 * >= the threshold half (NaN patterns compare false): exactly floor(65536 p) of the 65536 patterns are dropped for
 * p >= 254/65536 (tests/test_host_logic.py enumerates them). */
unsigned int step_tc_attn_drop_threshold(float drop_p);
/* ---- stage-1 (pre-training) attention on tcgen05, bf16 operands / fp32 accumulation and statistics, P <= 352 ----
 * Bytes of the log2-sum-exp buffer L [S, 4, P] fp32 the forward writes for the backward. */
size_t step_tc_attn_train_lse_bytes(int S, int P);
/* fp32 qkv rows [S*P, 288] (the in-projection output: q | k | v, head h at columns 24h..) -> the Q / K / V operand images
 * of step_tc_qkv (sizes from step_tc_attn_image_bytes; Q pre-scaled by log2(e)/sqrt(24); every pad row written as zero).
 * `bound` (may be NULL): the row-bound workspace step_tc_attention reads, filled as step_tc_qkv fills it. */
int step_tc_attn_train_pack(const float *qkv, int S, int P, void *q_img, void *k_img, void *v_img, float *bound, void *stream);
/* Training forward: out [S*P, 96] fp32 = dropout(softmax(q k^T / sqrt(24))) v per (sequence, head) and lse = the per-row
 * log2-sum-exp of the log2-domain scores.  Attention-probability dropout from the counter hash keyed by `seed`
 * (keep probability exactly 1 - floor(65536 p) / 65536, see step_tc_attn_train_keep_mask). */
int step_tc_attn_train_fwd(const void *q_img, const void *k_img, const void *v_img, int S, int P, float drop_p,
                           unsigned long long seed, float *out, float *lse, void *stream);
/* Training backward: dqkv [S*P, 288] fp32 (every column of every row written) from the images, the forward's out and lse,
 * and dout [S*P, 96]; the dropout mask is regenerated from (drop_p, seed). */
int step_tc_attn_train_bwd(const void *q_img, const void *k_img, const void *v_img, const float *out, const float *lse,
                           const float *dout, int S, int P, float drop_p, unsigned long long seed, float *dqkv, void *stream);
/* Test helper: mask [S, 4, P, P] uint8 = 1 where the forward and backward above keep the probability (query row, key column). */
int step_tc_attn_train_keep_mask(int S, int P, float drop_p, unsigned long long seed, unsigned char *mask, void *stream);
size_t step_ts_encoder_bf16_workspace_bytes(int B, int N, int P);
/* Whole encoder in bf16: series -> hidden [B,N,P,96] fp32 (same contract as step_ts_encoder_fwd). */
int step_ts_encoder_fwd_bf16(const float *series, long long sB, long long sT, long long sN, int B, int N, int P,
                             const float *patch_w, const float *patch_b, const float *pos,
                             const step_ts_layer_weights *h_layers, const step_ts_layer_images *h_images, int n_layers,
                             const float *final_norm_w, const float *final_norm_b, float *hidden, void *seq_img,
                             void *workspace, size_t workspace_bytes, float drop_p, unsigned long long seed, void *stream);
/* seq_img (optional output of step_ts_encoder_fwd_bf16, may be NULL): the hidden states once more as a per-sample
 * K-major bf16 image [B][P*12 chunks][R = round_up(N,128)][8] (row = node, K = (patch, feature)) - the operand of the
 * tensor-core Gram GEMM below. */
size_t step_tc_seq_image_bytes(int B, int N, int P);
/* Build the same image from fp32 hidden states [B,N,P,96] (node-sharded mode: after the all-gather). */
int step_tc_hidden_to_seq_image(const float *hidden, int B, int N, int P, void *seq_img, void *stream);
/* Cosine-similarity Gram matrix from the sequence image on tcgen05 (similarity.py:6-16; norms = sqrt of the Gram
 * diagonal).  gram_scratch, sim: [B,N,N] fp32. */
int step_tc_cosine_gram(const void *seq_img, int B, int N, int P, float *gram_scratch, float *sim, void *stream);

/* Node-sharded mode: raw Gram rows of the 128-row tiles tile_first, tile_first + tile_step, ... only (a rank's share; the
 * other rows of `gram` [B,N,N] are left untouched - a zero-initialised buffer summed over ranks is the full matrix), and
 * the normalisation sim = G / ((sqrt(G_ii)+1e-7)(sqrt(G_jj)+1e-7)) as a separate step after the exchange. */
int step_tc_gram_rows(const void *seq_img, int B, int N, int P, int tile_first, int tile_step, float *gram, void *stream);
int step_gram_normalize(const float *gram, int B, int N, float *sim, void *stream);

/* ------------------------------------------------------------------------ *
 * kNN prior graph: cosine-similarity Gram matrix + global top-k select
 *   step/step_arch/similarity.py:6-16,
 *   step/step_arch/discrete_graph_learning.py:91-111,164-166
 * ------------------------------------------------------------------------ */

/* x: [B, N, D] -> sim [B, N, N] = (x x^T) / ((|x_i|+1e-7)(|x_j|+1e-7)); norms: [B, N] scratch. */
int step_cosine_gram_f32(const float *x, int B, int N, long long D, float *norms, float *sim, void *stream);

/* adj[b,i,j] = 1 if sim[b,i,j] is among the k largest of the N*N entries of
 * sample b (ties at the threshold: lowest flat index first), is non-zero, and
 * i != j; else 0. */
int step_topk_mask_f32(const float *sim, int B, int N, int k, float *adj, void *stream);

/* ------------------------------------------------------------------------ *
 * Edge logits + hard Gumbel-softmax sample
 *   step/step_arch/discrete_graph_learning.py:11-45,148-161
 * ------------------------------------------------------------------------ */

/* logits[i,j,c] = fc_cat(relu(ut[:,j] + v[i,:]))[c] for the batch-invariant edge MLP.
 *   ut = (feat @ W_out[:, :100]^T)^T  [100, N]  (sender half, transposed),
 *   v  =  feat @ W_out[:, 100:]^T + b_out  [N, 100]  (receiver half + bias).
 * theta[i,j] = softmax(logits[i,j,:])[0]  (step/step_arch/step.py:72). */
int step_edge_logits_fwd(const float *ut, const float *v, const float *cat_w /*[2,100]*/, const float *cat_b /*[2]*/,
                         int N, int F, float *logits /*[N,N,2]*/, float *theta /*[N,N]*/, void *stream);

/* Backward of step_edge_logits_fwd.  dlogits: [N,N,2].  Outputs (overwritten):
 * dut [F,N], dv [N,F], dcat_w [2,F], dcat_b [2]. */
int step_edge_logits_bwd(const float *dlogits, const float *ut, const float *v, const float *cat_w,
                         int N, int F, float *dut, float *dv, float *dcat_w, float *dcat_b, void *stream);

/* sampled[b,i,j] in {0,1}: class-0 indicator of the hard Gumbel-softmax sample at
 * temperature tau with Gumbel noise g = -log(-log(U+1e-10)+1e-10), diagonal forced to 0.
 * y0[b,i,j]: the soft class-0 probability (saved for the straight-through backward).
 * uniform: [B, N*N, 2] externally supplied U(0,1) draws (parity / injection), or NULL to
 * draw them in-kernel from the counter-based generator keyed by `seed`. */
int step_gumbel_sample_fwd(const float *logits /*[N,N,2]*/, const float *uniform, int B, int N, float tau,
                           unsigned long long seed, float *sampled, float *y0, void *stream);

/* dlogits[i,j,0] = sum_b dsampled[b,i,j] * y0 (1 - y0) / tau (0 on the diagonal), dlogits[i,j,1] = -dlogits[i,j,0];
 * if accumulate != 0 the result is added to dlogits. */
int step_gumbel_sample_bwd(const float *dsampled, const float *y0, int B, int N, float tau, int accumulate,
                           float *dlogits, void *stream);


/* ------------------------------------------------------------------------ *
 * STEP loss, value + gradients in one call
 *   step/step_loss/step_loss.py:5-16 + basicts/metrics/mae.py:5-28 + basicts/data/transform.py:48-65
 *   loss = masked_mae(pred*std+mean, real*std+mean, null_val) + coeff * BCE(theta, adj_knn)
 * pred/real: n_pred values of the selected target feature (unscaled); theta: [N,N] (batch-invariant);
 * adj_knn: [B,N,N].  use_nan_mask != 0 <=> null_val is NaN.  Outputs: loss [1], dpred [n_pred] (w.r.t. the unscaled
 * prediction), dtheta [N,N].  scratch: >= 64 bytes.
 * ------------------------------------------------------------------------ */
int step_loss_fwd_bwd(const float *pred, const float *real, long long n_pred, float mean, float stdv, float null_val,
                      int use_nan_mask, const float *theta, const float *adj_knn, int B, int N, float coeff, float *loss,
                      float *dpred, float *dtheta, void *scratch, void *stream);

/* ------------------------------------------------------------------------ *
 * Discrete graph learning: convolutional part of the batch-invariant "global feature" trunk
 *   step/step_arch/discrete_graph_learning.py:131-133
 *   x [N, L0] -> Conv1d(1,8,10) -> ReLU -> BN(8) -> Conv1d(8,16,10) -> ReLU -> BN(16) -> y2n [N, 16, L0-18]
 * y1 is never materialised (recomputed from x wherever needed).  bnK_stats: [4][C] = mean, biased var,
 * scale, shift - written when training != 0 (batch statistics), read as given when training == 0.
 * y2: pre-BN2 conv output kept for the backward pass.  scratch: >= 4096 bytes.
 * ------------------------------------------------------------------------ */
int step_dgl_conv_fwd(const float *x, int N, int L0, const float *w1, const float *b1, const float *g1, const float *be1,
                      const float *w2, const float *b2, const float *g2, const float *be2, float eps, int training,
                      float *bn1_stats, float *bn2_stats, float *y2, float *y2n, void *scratch, void *stream);
/* Backward of step_dgl_conv_fwd (training mode).  dy2n: [N,16,L0-18].  dy1n_scratch: [N,8,L0-9] floats.
 * Outputs (overwritten): dw1 [8,1,10], db1 [8], dg1/dbe1 [8], dw2 [16,8,10], db2 [16], dg2/dbe2 [16]. */
int step_dgl_conv_bwd(const float *dy2n, const float *x, int N, int L0, const float *w1, const float *b1, const float *g1,
                      const float *w2, const float *g2, float eps, const float *bn1_stats, const float *bn2_stats,
                      const float *y2, float *dy1n_scratch, float *dw1, float *db1, float *dg1, float *dbe1, float *dw2,
                      float *db2, float *dg2, float *dbe2, void *scratch, void *stream);

/* ------------------------------------------------------------------------ *
 * Discrete graph learning: dense part of the trunk, feat = BN3(relu(y2n W^T + b))  [N,100]
 *   step/step_arch/discrete_graph_learning.py:66,134-135 (self.fc, self.bn3; BatchNorm1d over the N nodes)
 * The three GEMMs (forward, dX, dW) run on tcgen05 with split-bf16 operands (fp32-class accuracy) and stream
 * y2n / fc.weight exactly once.  [k_begin, k_end) selects the slice of the K axis this call covers (the whole
 * [0, K) on one GPU; a rank's shard when the trunk is partitioned): x and w are always the full row-major
 * matrices with row stride K.
 * ------------------------------------------------------------------------ */
/* Number of split-K partials step_dgl_fc_fwd writes: partial must hold splits * N * 100 floats. */
int step_dgl_fc_splits(int N, long long k_begin, long long k_end);
/* z_raw[n][j] = sum_{k in range} x[n][k] w[j][k]   (no bias: a sharded caller all-reduces z_raw first). */
int step_dgl_fc_fwd(const float *x /*[N,K]*/, const float *w /*[100,K]*/, int N, long long K, long long k_begin,
                    long long k_end, float *partial, float *z_raw /*[N,100]*/, void *stream);
/* z = z_raw + bias (in place), feat = BN(relu(z)).  stats [3][100] = mean, biased var, rstd: written when
 * training != 0 (batch statistics over the N nodes); when training == 0 rows 0/1 hold the running statistics. */
int step_dgl_fc_bn_fwd(float *z, const float *bias, const float *gamma, const float *beta, int N, float eps, int training,
                       float *stats, float *feat /*[N,100]*/, void *stream);
/* Backward of step_dgl_fc_bn_fwd (training mode): g = dL/dz_raw [N,100], dgamma/dbeta/dbias [100]. */
int step_dgl_fc_bn_bwd(const float *dfeat, const float *z, const float *gamma, const float *stats, int N, float *g,
                       float *dgamma, float *dbeta, float *dbias, void *stream);
/* dx[n][k] = sum_j g[n][j] w[j][k],  dw[j][k] = dw_scale * sum_n g[n][j] x[n][k]   for k in [k_begin, k_end)
 * (k_begin a multiple of 64; entries outside the range are left untouched). */
int step_dgl_fc_bwd(const float *g, const float *x, const float *w, int N, long long K, long long k_begin, long long k_end,
                    float dw_scale, float *dx /*[N,K]*/, float *dw /*[100,K]*/, void *stream);

/* ------------------------------------------------------------------------ *
 * General fp32 GEMM on tcgen05 with split-bf16 operands (fp32-class accuracy) for the mid-size dense products the
 * reference runs through nn.Linear / Conv2d(1x1) / torch.matmul on cuBLAS:
 *   Graph WaveNet epilogue fc_his / end_conv_1 / end_conv_2 (graphwavenet/model.py:215-220), the fc_out halves of
 *   discrete graph learning (discrete_graph_learning.py:148-151), TSFormer pre-training backward (tsformer.py:71-160).
 *   C[M,N] (+)= alpha * sum_k opA(m,k) opB(n,k) [+ bias[n]] [epilogue]
 *   transA == 0: A row-major [M][K];  transA != 0: A row-major [K][M]
 *   transB == 0: B row-major [N][K] (an nn.Linear weight);  transB != 0: B row-major [K][N]
 *   epilogue 0 none, 1 ReLU, 2 mask: C = acc * (aux > 0), 3: C = relu(relu(acc + bias) + aux), aux_out = relu(acc + bias)
 *   ksplit > 1: the K range is split over grid.z and accumulated with fp32 atomics (epilogue 0 only).
 * ------------------------------------------------------------------------ */
int step_gemm_f32(const float *A, long long lda, int transA, const float *B, long long ldb, int transB, int M, int N, int K,
                  float alpha, const float *bias, int epilogue, const float *aux, long long ldaux, float *aux_out, int accumulate,
                  int ksplit, float *C, long long ldc, void *stream);
/* out[n] = sum_m x[m][n]  (bias gradients);  dz = dy * (y > 0)  (ReLU backward). */
int step_colsum_f32(const float *x, long long M, int N, long long ld, float *out, void *stream);
int step_relu_bwd_f32(const float *dy, const float *y, long long n, float *dz, void *stream);

/* ------------------------------------------------------------------------ *
 * Graph WaveNet prologue, forward + backward   step/step_arch/graphwavenet/model.py:121-130,144-166
 * ------------------------------------------------------------------------ */
/* x0 [B,T+1,N,32] = start_conv(left-padded history[..., 0:2]); history [B,T,N,C], w [32,2], bias [32]. */
int step_gw_start_fwd(const float *history, int B, int T, int N, int C, const float *w, const float *bias, float *x0, void *stream);
/* dw_db [96] = (dW [32,2] | db [32]) from dx0 [B,T+1,N,32]. */
int step_gw_start_bwd(const float *history, int B, int T, int N, int C, const float *dx0, float *dw_db, void *stream);
/* P1 = D^-1 (A + I), P2 = D'^-1 (A^T + I) for adj [B,N,N]; deg [2,B,N] (row / column degrees + 1) is kept for backward. */
int step_gw_supports_fwd(const float *adj, int B, int N, float *deg, float *P1, float *P2, void *stream);
/* dadj [B,N,N] from dP1, dP2; dots: [2,B,N] scratch. */
int step_gw_supports_bwd(const float *dP1, const float *dP2, const float *P1, const float *P2, const float *deg, int B, int N,
                         float *dots, float *dadj, void *stream);
/* P3 [N,N] = softmax_row(relu(E1 E2)), E1 [N,R], E2 [R,N] (R = 10). */
int step_gw_adp_fwd(const float *E1, const float *E2, int N, int R, float *P3, void *stream);
/* dE1 [N,R], dE2 [R,N] from dP3; scratch: [N,N] floats. */
int step_gw_adp_bwd(const float *E1, const float *E2, const float *P3, const float *dP3, int N, int R, float *scratch, float *dE1,
                    float *dE2, void *stream);

/* ------------------------------------------------------------------------ *
 * Graph WaveNet layer stack (8 x gated dilated conv + skip + diffusion GCN + BN)
 *   step/step_arch/graphwavenet/model.py:169-213 (+ gcn :35-48, nconv :10-16)
 * Activation layout is [B, T, N, 32] (channels innermost).
 * ------------------------------------------------------------------------ */
typedef struct step_gw_layer_params {
  const float *filter_w; /* [32,32,1,2] */
  const float *filter_b; /* [32] */
  const float *gate_w;   /* [32,32,1,2] */
  const float *gate_b;   /* [32] */
  const float *skip_w;   /* [256,32] */
  const float *skip_b;   /* [256] */
  const float *mlp_w;    /* [32,224]  (NULL for the last layer: its gcn output is dead, model.py:217-218) */
  const float *mlp_b;    /* [32] */
  const float *bn_w;     /* [32] */
  const float *bn_b;     /* [32] */
} step_gw_layer_params;

typedef struct step_gw_layer_grads {
  float *filter_w, *filter_b, *gate_w, *gate_b, *skip_w, *skip_b, *mlp_w, *mlp_b, *bn_w, *bn_b;
} step_gw_layer_grads;

/* Size in floats of the activation stash / scratch the stack needs. */
size_t step_gwnet_stash_floats(int B, int N, int n_layers);

/* Forward of the layer stack.
 *   x0:       [B, 13, N, 32]   start_conv output (model.py:155)
 *   supports: P1,P2 [B,N,N] (random-walk normalised sampled graph and its transpose-graph,
 *             model.py:160), P3 [N,N] (adaptive adjacency, model.py:165)
 *   skip_out: [B, N, 256]  sum over layers of the skip conv at the last time step (the only
 *             column that survives the reference's truncation `skip[..., -T:]`, model.py:188-192)
 *   bn_stats: [n_layers, 4, 32] per layer (mean, biased var, scale, shift) of the batch statistics
 *             when training != 0; when training == 0 the caller pre-fills scale/shift from the running
 *             statistics and they are used as is.
 *   stash:    activations kept for the backward pass (step_gwnet_stash_floats).
 *   drop_p/seed: dropout on the gcn output (model.py:47) when training != 0. */
int step_gwnet_stack_fwd(const float *x0, const float *P1, const float *P2, const float *P3,
                         const step_gw_layer_params *h_layers, int n_layers, int B, int N,
                         int training, float drop_p, unsigned long long seed,
                         float *skip_out, float *bn_stats, float *stash, void *stream);

/* Backward of the layer stack (training mode), to be called after step_gwnet_stack_fwd on the same stash (which
 * holds z, f, g, q_s and - on the tensor-core mix path - a_s of every layer).  dskip: [B,N,256].  P1t/P2t/P3t are the
 * transposed supports.  Outputs: dx0 [B,13,N,32], dP1,dP2 [B,N,N], dP3 [N,N], per-layer
 * parameter gradients (all overwritten). */
int step_gwnet_stack_bwd(const float *dskip, const float *x0, const float *P1, const float *P2, const float *P3,
                         const float *P1t, const float *P2t, const float *P3t,
                         const step_gw_layer_params *h_layers, const step_gw_layer_grads *h_grads, int n_layers,
                         int B, int N, float drop_p, unsigned long long seed,
                         const float *bn_stats, float *stash, float *dx0, float *dP1, float *dP2, float *dP3,
                         void *stream);

/* ------------------------------------------------------------------------ *
 * Optimiser step + metric accumulation (SURVEY section 8(f).2)
 *   clip_grad_norm_(max_norm) + torch.optim.Adam(lr, betas, eps, weight_decay) - step/STEP_METR-LA.py:88-107 - over all
 *   parameter tensors in two launches; masked MAE / RMSE / MAPE accumulated on the device (base_tsf_runner.py:252-254
 *   syncs the host three times per step for them).
 * Tables (device memory, int64 unless noted): p_ptr / g_ptr = addresses of parameter i and of its gradient (0 = no
 * gradient this step: the tensor is skipped), numel, state_off = offset of tensor i in the flat moment buffers m / v;
 * chunk_tensor (int32) / chunk_off: one entry per block of step_opt_chunk_elems() elements.
 * steps_in / steps_out (int32 per tensor, two distinct buffers the caller swaps every call): Adam steps taken so far -
 * torch keeps `step` per parameter, a tensor without gradient does not advance.
 * sumsq: 1 double scratch; norm_out (optional): the gradient norm before clipping.
 * ------------------------------------------------------------------------ */
int step_opt_chunk_elems(void);
int step_clip_adam_step(const long long *p_ptr, const long long *g_ptr, const long long *numel, const long long *state_off,
                        const int *chunk_tensor, const long long *chunk_off, int n_chunks, const int *steps_in, int *steps_out,
                        float *m, float *v, double *sumsq, float max_norm, float lr, float beta1, float beta2, float eps,
                        float weight_decay, float *norm_out, void *stream);
/* Adds this batch's masked MAE / RMSE / MAPE (of pred*std+mean vs real*std+mean, null handling of basicts/metrics) to
 * acc[0..2] and 1 to acc[3]; sums[5] is scratch that must be zero before the first call. */
int step_metrics_accumulate(const float *pred, const float *real, long long n, float mean, float stdv, float null_val,
                            int use_nan_mask, double *sums, double *acc, void *stream);

/* Test hook: the dropout site of the gcn output (graphwavenet/model.py:47) applied to a stand-alone [rows, 32] buffer with
 * exactly the mask the layer kernels draw for elements [0, rows*32) of layer `layer`. */
int step_gwnet_dropout_probe(const float *x, long long rows, float drop_p, unsigned long long seed, int layer, float *y,
                             void *stream);

#ifdef __cplusplus
}
#endif
#endif /* STEP_B200_H_ */
