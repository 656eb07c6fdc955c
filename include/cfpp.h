/* cfpp.h -- C ABI of libcfpp.so: B200 (sm_100a) kernels for the ContextFlow++ flow log-density path.
 *
 * The reference (gudovskiy/contextflow) has no FFI: its hot path is the Python class API
 * FlowLayer.forward(x, context) -> (z, ldj) (contextflow/layers/flowlayer.py:7-24) evaluated by PyTorch eager ops.
 * This header is the boundary a binding replaces that path with; each entry point cites the reference
 * code it computes.  Conventions:
 *   - every pointer is a DEVICE pointer owned by the caller (torch allocates); fp32 NCHW contiguous unless a
 *     batch stride argument says otherwise; contexts are int64 (B, n_ctx);
 *   - `stream` is a cudaStream_t passed as void*; launches are asynchronous on it;
 *   - return value: 0 = ok, non-zero = error (message via cfpp_last_error(), thread-local); nothing is thrown
 *     across the ABI and the library never exits the process; no global mutable state.
 * File paths below are relative to /root/reference/contextflow.
 */
#ifndef CFPP_H_
#define CFPP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CFPP_OK 0
#define CFPP_ERR_ARG 1
#define CFPP_ERR_CUDA 2
#define CFPP_ERR_UNSUPPORTED 3

int cfpp_version(void);
const char* cfpp_last_error(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches claim) */
int64_t cfpp_launch_count(void);
/* asynchronous copy of `bytes` between devices of this process on `stream` (a stream of the CURRENT device): single-process N-GPU
 * log_prob pulls a batch slice to / pushes its (b, M) result from the device that scores it (contextflow_b200/multigpu.py) */
int cfpp_copy_peer_async(void* dst, int dst_device, const void* src, int src_device, int64_t bytes, void* stream);

/* ---- index-only layers (bit exact) ------------------------------------------------------------------ */
/* Squeeze.forward, layers/squeeze.py:10-11: y[b,(c p1 p2),h,w] = x[b,c,h*p1+i,w*p2+j]; (H,W) are INPUT dims. */
int cfpp_squeeze_fwd(const float* x, float* y, int B, int C, int H, int W, int p1, int p2, void* stream);
/* the same over the first C channels of every sample of a wider tensor (batch stride x_bstride floats): SplitPrior's z = x[:, :C]
 * (splitprior.py:13) feeding the next block's Squeeze without a copy of its own; 2x2, W % 8 == 0 only (CFPP_ERR_UNSUPPORTED otherwise) */
int cfpp_squeeze_strided_fwd(const float* x, int64_t x_bstride, float* y, int B, int C, int H, int W, int p1, int p2, void* stream);
/* Squeeze.reverse, layers/squeeze.py:13-14; (H,W) are the dims of the un-squeezed OUTPUT. */
int cfpp_squeeze_inv(const float* y, float* x, int B, int C, int H, int W, int p1, int p2, void* stream);
/* PermuteAxes((0,2,1,3)).forward, layers/permute_axes.py:13-14: y[b,h,c,w] = x[b,c,h,w]. */
int cfpp_permute_fwd(const float* x, float* y, int B, int C, int H, int W, void* stream);
/* channel slice copy: y[b, 0:Cn, :] = x[b, c0:c0+Cn, :]  (SplitPrior's x[0], layers/splitprior.py:13-15). */
int cfpp_slice_channels(const float* x, float* y, int B, int C, int HW, int c0, int Cn, void* stream);

/* the adjoint of cfpp_slice_channels: dst[b, c0:c0+Cn, :] = src[b, 0:Cn, :] (SplitPrior backward); other channels untouched. */
int cfpp_place_channels(const float* src, float* dst, int B, int C, int HW, int c0, int Cn, void* stream);

/* ---- data format in front of the path: SURVEY §8(f)-4 ----------------------------------------------------------- */
/* Sliding windows over a raw multivariate series, generated on the device in the model's input layout: get_windows
 * (datasets/mtad_data_preprocess.py:58-74: window ending at row e covers rows e-L+1..e, rows before 0 replicate row 0) followed by
 * the transpose / float32 cast of sliding_window_dataset (datasets/mtad_dataloader.py:106-110):
 *   x[b, d, t, 0] = (float) ts[max(0, e_b - L + 1 + t), d],  e_b = end[b] (int64, device) or end0 + b * stride when end == NULL.
 * ts: (n_rows, D) row-major, float32 or float64 (ts_is_f64).  Bit exact (index work + the IEEE float64 -> float32 rounding torch applies). */
int cfpp_windows_fwd(const void* ts, int ts_is_f64, const int64_t* end, int64_t end0, int64_t stride, float* x,
                     int B, int64_t n_rows, int D, int L, void* stream);

/* ---- image prologue ----------------------------------------------------------------------------------- */
/* Dequantization.forward, layers/dequantize.py:14-17: y = x + u. */
int cfpp_add_fwd(const float* x, const float* u, float* y, int64_t n, void* stream);
/* Normalization.forward (scalar scale), layers/normalize.py:27-34: y = x / scale + translation. */
int cfpp_normalize_fwd(const float* x, float* y, int64_t n, float scale, float translation, void* stream);
/* LogitTransform.forward/logdet, layers/transforms.py:11-18: y = log x - log(1-x); ldj[b] = sum(-log x - log(1-x)). */
int cfpp_logit_fwd(const float* x, float* y, float* ldj, int B, int n_per_sample, void* stream);
/* Augment.forward + StandardNormal.log_prob, layers/augment.py:14-18, distributions/gaussian.py:50-72:
 * y = cat([x, eps], 1) with eps (B,A,HW); ldj[b] = sum(0.5 log 2pi + 0.5 eps^2). */
int cfpp_augment_fwd(const float* x, const float* eps, float* y, float* ldj, int B, int C, int A, int HW, void* stream);
/* The four prologue layers of create_model (model.py:97-100) + optional Augment, in one pass:
 * v = ((x+u)/s0 + t0)/s1 + t1; y = logit(v) (C channels) ++ eps (A channels, may be 0);
 * ldj[b] = ldj_const + sum(-log v - log(1-v)) + sum(0.5 log 2pi + 0.5 eps^2). */
int cfpp_prologue_fwd(const float* x, const float* u, const float* eps, float* y, float* ldj, int B, int C, int A, int HW,
                      float s0, float t0, float s1, float t1, float ldj_const, void* stream);

/* ---- invertible 1x1 conv and ActNorm ------------------------------------------------------------------- */
/* torch.slogdet(NN)[1], layers/conv1x1.py:43,53: log|det A| of a DxD matrix (fp64 LU inside), D <= 128. */
int cfpp_slogdet(const float* A, int D, float* logabsdet, void* stream);
/* Conv1x1.forward, layers/conv1x1.py:28-57.
 *   c == NULL : z = NN x per pixel; ldj[b] = HW * logabsdet.
 *   c != NULL : c is the raw CN output (B,D,D); W_b = tril(c,-1) + diag(exp(diag c)) [- I + NN if contextflow];
 *               ldj[b] = HW * ((contextflow ? logabsdet : 0) + sum diag c_b) + HW * logp_c[b].
 * Optional fused ActNorm epilogue (t, logs non-NULL; an_per_sample 0: shared (D) vectors; 1: per-sample (B,D) arrays;
 * 2: one (B,2D) array 'b (p d)' as ActNorm.CN produces it -- an_t points at it and an_logs = an_t + D):
 *   z = (z - t) * exp(-logs); ldj[b] += sum_d logs (+ an_logp_scale * an_logp_c[b]).   (layers/actnorm.py:37-60) */
int cfpp_conv1x1_fwd(const float* x, float* z, float* ldj, const float* NN, const float* logabsdet,
                     const float* c, const float* logp_c, int contextflow,
                     const float* an_t, const float* an_logs, int an_per_sample, const float* an_logp_c, float an_logp_scale,
                     int B, int D, int HW, void* stream);
/* Conv1x1.forward with a context_net, layers/conv1x1.py:31-50, INCLUDING its context network `c = self.CN(c)` (:33) and the optional
 * ActNorm epilogue (layers/actnorm.py:37-60) in one persistent kernel: the (B,D,D) matrix c never exists in HBM.
 *   e        (B,K)  encoder output of the layer's context_net (K = context_net.C <= 64);
 *   cnw_tri  (K,T)  CN.weight restricted to the lower triangle + diagonal, K-major: cnw_tri[k][i(i+1)/2 + j] = CN.weight[i*D + j][k], j <= i,
 *                   T = D(D+1)/2 (the strictly upper entries of c are discarded by torch.tril, conv1x1.py:36,40,46);
 *   cnb_tri  (T)    CN.bias in the same order.
 * W_b, ldj and the epilogue exactly as cfpp_conv1x1_fwd with c != NULL; an_per_sample must be 1 or 2 when an_t is given.
 * cfpp_conv1x1_ctx_supported: 1 when (D, HW, K) has a plan (D <= 128, HW % 4 == 0, the tiles fit shared memory); otherwise callers use
 * cfpp_cn_batch + cfpp_conv1x1_fwd. */
int cfpp_conv1x1_ctx_supported(int B, int D, int HW, int K);
int cfpp_conv1x1_ctx_fwd(const float* x, float* z, float* ldj, const float* e, const float* cnw_tri, const float* cnb_tri,
                         const float* NN, const float* logabsdet, const float* logp_c, int contextflow,
                         const float* an_t, const float* an_logs, int an_per_sample, const float* an_logp_c, float an_logp_scale,
                         int B, int D, int HW, int K, void* stream);
/* ActNorm.forward, layers/actnorm.py:37-60: t,logs = base (D) [+ c (B,2D) 'b (p d)'] per mode:
 *   mode 0: base only; mode 1: base + c (contextflow); mode 2: c only (conventional).
 * z = (x - t) * exp(-logs); ldj[b] = sum_d logs[b,d] + logp_scale * logp_c[b]   (note: no H*W factor, App. C-1). */
int cfpp_actnorm_fwd(const float* x, float* z, float* ldj, const float* base_t, const float* base_logs, const float* c,
                     const float* logp_c, float logp_scale, int mode, int B, int D, int HW, void* stream);
/* ActNorm.initialize, layers/actnorm.py:28-35: mean[d], logstd[d] = log(unbiased std + 1e-8) over (B,HW). */
int cfpp_actnorm_stats(const float* x, float* mean, float* logstd, int B, int D, int HW, void* stream);

/* ---- coupling -------------------------------------------------------------------------------------------- */
/* The fused memory-bound coupling transform, layers/coupling.py:50-66 (also :131-148):
 *   t = h[:, :C/2] (+ add[:, :C/2]); r = h[:, C/2:] (+ add[:, C/2:]); log_s = 2 tanh(r/2);
 *   z = cat(x[:, :C/2], x[:, C/2:] * exp(log_s) + t); ldj[b] = sum log_s + logp_scale * logp_c[b].
 * add (B,C) and logp_c (B) may be NULL.  One HBM pass: reads x,h once, writes z once (12*C*HW bytes/sample). */
int cfpp_coupling_fwd(const float* x, const float* h, const float* add, const float* logp_c, float logp_scale,
                      float* z, float* ldj, int B, int C, int HW, void* stream);
/* Coupling.NN, layers/coupling.py:26-29: Conv(Cin->Ch,1x1) ReLU Conv(Ch->Ch, KHxKW, reflect pad (KH/2,KW/2)) ReLU
 * Conv(Ch->Cout,1x1).  x is (B, >=Cin, H, W) with batch stride x_bstride (the coupling's x0 half is read in place).
 * Weights are PACKED K-major: w1t (Cin,Ch), w2t (Ch*KH*KW, Ch) with k = (cin*KH+ky)*KW+kx, w3t (Ch,Cout).
 * bias1_b (B,Ch) optional per-sample first-layer bias replacing b1 (conventional context concat, coupling.py:47). */
int cfpp_conv_cond_fwd(const float* x, int64_t x_bstride, float* h,
                       const float* w1t, const float* b1, const float* bias1_b,
                       const float* w2t, const float* b2, const float* w3t, const float* b3,
                       int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, void* stream);

/* The same conditioner on the tcgen05 tensor cores (kind::tf32, fp32-faithful 3xTF32 split, TMEM accumulators, weights streamed
 * by bulk TMA copies; contextflow_b200/csrc/conv_cond_tc.cu).  Weights are repacked ONCE per parameter version by
 * cfpp_conv_cond_tc_pack from the torch layouts: w1 (Ch, >=Cin) with row stride w1_stride, w2 (Ch, Ch, KH, KW), w3 (Cout, Ch);
 * b1/b2/b3 are the plain bias vectors.  Supported: Ch % 16 == 0, 16 <= Ch <= 128, Cin <= 64 (32 for the tf32 kind), Cout <= 128, KH,KW in {1,3},
 * (Cin*H*W) % 4 == 0, x_bstride % 4 == 0, x 16-byte aligned -- cfpp_conv_cond_tc_supported() answers for a shape; other shapes
 * use cfpp_conv_cond_fwd (CFPP_ERR_UNSUPPORTED is returned, nothing is launched). */
int64_t cfpp_conv_cond_tc_pack_bytes(int Cin, int Ch, int Cout, int KH, int KW);   /* -1 when unsupported */
int cfpp_conv_cond_tc_pack(const float* w1, int w1_stride, const float* w2, const float* w3, void* out,
                           int Cin, int Ch, int Cout, int KH, int KW, void* stream);
int cfpp_conv_cond_tc_supported(int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, int64_t x_bstride);
int cfpp_conv_cond_tc_fwd(const float* x, int64_t x_bstride, float* h, const void* wpack,
                          const float* b1, const float* bias1_b, const float* b2, const float* b3,
                          int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, void* stream);
/* Training forward of the conditioner (coupling.py:26-29 under autograd): h as cfpp_conv_cond_tc_fwd plus the post-ReLU activations
 * a1 = relu(W1 x0 + b1), a2 = relu(W2 * a1 + b2) as fp32 (B, Ch, H, W), which the backward pass reads (ReLU masks, weight gradients). */
int cfpp_conv_cond_tc_train_fwd(const float* x, int64_t x_bstride, float* h, float* a1, float* a2, const void* wpack,
                                const float* b1, const float* bias1_b, const float* b2, const float* b3,
                                int B, int Cin, int Ch, int Cout, int H, int W, int KH, int KW, void* stream);
/* The conditioner and the affine coupling transform it feeds (coupling.py:39-66) in ONE kernel: the conditioner output h never reaches
 * HBM.  x, z (B, C, H, W) contiguous; x0 = x[:, :C/2] is the conditioner input, h = NN(x0) (+ add[b, :] per channel: CN(c), additive
 * contextflow conditioning, coupling.py:45; NULL: none; bias1_b as in cfpp_conv_cond_tc_fwd for the concatenated form);
 * t = h[:, :C/2], log_s = 2 tanh(h[:, C/2:] / 2); z = cat(x0, x1 * exp(log_s) + t); ldj[b] = sum log_s + logp_scale * logp_c[b].
 * Weights as packed by cfpp_conv_cond_tc_pack(Cin = C/2, Cout = C).  C % 16 == 0; cfpp_conv_cond_tc_coupling_supported answers for a shape. */
int cfpp_conv_cond_tc_coupling_supported(int B, int C, int Ch, int H, int W, int KH, int KW);
int cfpp_conv_cond_tc_coupling_fwd(const float* x, float* z, float* ldj, const void* wpack, const float* b1, const float* bias1_b,
                                   const float* b2, const float* b3, const float* add, const float* logp_c, float logp_scale,
                                   int B, int C, int Ch, int H, int W, int KH, int KW, void* stream);
/* Operand arithmetic of the tensor-core conditioner in this process: 1 (default) = scaled fp16 hi/lo pairs, tcgen05 kind::f16
 * (22+ significand bits, values saturate at +-65504); 0 = tf32 hi/lo pairs, kind::tf32 (fp32 range; environment
 * CFPP_TC_KIND=tf32).  Packed weights are specific to the kind they were packed under. */
int cfpp_conv_cond_tc_kind(void);
/* geometry of the last cfpp_conv_cond_tc_fwd launch (tests / bench): {segment layout, samples per tile, stored rows, M-tiles of
 * stage 1, M-tiles of stages 2-3, ring stages, shared-memory bytes, tiles, CTAs resident per SM, operand row bytes, software-pipelined
 * tiles (1/0)} (11 ints; pass room for 12) */
void cfpp_conv_cond_tc_last_plan(int* out12);
/* debug instrumentation: device array of 12 int64 cycle counters that CTA 0 accumulates over its tiles; NULL = off.
 * epilogue thread 0: {wait x0, x0 transform, wait stage-1 MMAs, epilogue 1, wait stage-2 MMAs, epilogue 2, wait stage-3 MMAs,
 * epilogue 3}; MMA thread: {wait weight chunk, issue, wait operands, spare} */
void cfpp_conv_cond_tc_set_profile(void* counters8);

/* SimpleViT conditioner of TransCoupling, layers/simple_vit.py:91-127 (heads=1, dim_head=64, dim=mlp_dim=T, GELU-erf,
 * LayerNorm eps 1e-5).  All weight matrices PACKED K-major (in_features, out_features). */
typedef struct {
  int Cin, H, W, p1, p2;     /* input channels (x0 half, or + concat), image size, patch size */
  int T, depth, n_tok, patch_dim;
  const float *ln0_w, *ln0_b;              /* LayerNorm(patch_dim) */
  const float *pe_wt, *pe_b;               /* Linear(patch_dim -> T) */
  const float *ln1_w, *ln1_b;              /* LayerNorm(T) */
  const float *pos;                        /* (n_tok, T) sincos table (simple_vit.py:18-27) */
  const float *lnf_w, *lnf_b;              /* transformer.norm */
  const float* layers;                     /* depth x per-layer block, see cfpp_vit_layer_floats() */
} cfpp_vit_desc;
/* Packed matrices have their output dimension zero-padded to NP = 16*ceil(T/16) columns (pe_wt, Wo, W1, W2; biases too).
 * floats per packed layer block: [ln_a w,b (2T)] [Wqkv^T (T*192)] [Wo^T (64*NP)] [ln_f w,b (2T)] [W1^T (T*NP)] [b1 (NP)] [W2^T (T*NP)] [b2 (NP)] */
int64_t cfpp_vit_layer_floats(int T);
/* h (B, T/(p1 p2), H, W).  extra (B, Cextra) optional per-sample constant channels appended to x0 (conventional concat). */
int cfpp_vit_cond_fwd(const float* x, int64_t x_bstride, const float* extra, int Cextra, float* h,
                      const cfpp_vit_desc* desc, int B, void* stream);

/* The same conditioner on the tensor cores (csrc/vit_tc.cu) for token widths T <= 64, patch_dim <= 64, n_tok dividing 32 and no
 * concatenated context channels (the SMAP stack: T = 52, 4 tokens): thread = token row with the residual stream in registers, every
 * linear layer a 128 x 64 x 64 tcgen05.mma group on fp16 hi / scaled-lo operand pairs (fp32-faithful, as the conv conditioner).
 * Weights: cfpp_vit_tc_pack_bytes(depth) bytes holding 1 + 6*depth chunks in the order patch-embedding, then per layer q, k, v
 * (rows 0-63 / 64-127 / 128-191 of to_qkv.weight), to_out, mlp[1], mlp[3]; each chunk written by cfpp_vit_tc_pack_chunk from the
 * row-major nn.Linear weight (out_features = n_rows <= 64, in_features = k_cols <= 64, leading dimension ld).  LayerNorm parameters,
 * biases and the positional table are read from the descriptor exactly as cfpp_vit_cond_fwd reads them. */
int cfpp_vit_tc_supported(int T, int patch_dim, int n_tok, int Cextra);
int64_t cfpp_vit_tc_pack_bytes(int depth);
int cfpp_vit_tc_pack_chunk(const float* w, int ld, int n_rows, int k_cols, void* out_chunk, void* stream);
int cfpp_vit_tc_fwd(const float* x, int64_t x_bstride, float* h, const cfpp_vit_desc* desc, const void* wpack, int B, void* stream);

/* General form (csrc/vit_tc2.cu): T <= 192 (T % 4 == 0), any token count up to 128 per sample, no concatenated context channels (the
 * ATM stack: T in {36, 72, 144, 152}).  Four threads per token row, P = ceil(T/64) operand panels; the weight stream holds
 * cfpp_vit_tc2_chunks() chunks of the cfpp_vit_tc_pack_chunk format, one per (64-row output block n, 64-column input block p) of a
 * matrix, n outer / p inner, matrices in the order patch-embedding, then per layer to_qkv (192 x T), to_out (T x 64), mlp[1], mlp[3]. */
int cfpp_vit_tc2_supported(int T, int patch_dim, int n_tok, int Cextra);
int64_t cfpp_vit_tc2_chunks(int T, int patch_dim, int depth);
int cfpp_vit_tc2_fwd(const float* x, int64_t x_bstride, float* h, const cfpp_vit_desc* desc, const void* wpack, int B, void* stream);

/* ---- Gaussian-mixture log-prob ----------------------------------------------------------------------------- */
/* GaussianMixtureDistribution.log_prob, layers/distributions/gaussian.py:142-161 (torch.distributions semantics):
 * out[b,m] = logsumexp_k( logmix[m,k] + sum_e N(x[b,e]; mG[m,k,e] (+cm), softplus(sG[m,k,e] (+cs))) ) + logp_scale*logp_c[b]
 * with e over (d,h,w), logmix = log_softmax(log(clamp(softmax(wG)/sum, eps, 1-eps))).
 * ctx_off (B, 2*M*K*D) optional: 'b (p m k d)' mean / pre-softplus-scale offsets per sample. x has batch stride. */
int cfpp_gmm_logprob(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* wG,
                     const float* ctx_off, const float* logp_c, float logp_scale, float* out, float* workspace,
                     int B, int M, int K, int D, int HW, void* stream);
/* floats of caller-provided scratch cfpp_gmm_logprob needs (hoisted 1/(2 sigma^2) table + per-component constants) */
int64_t cfpp_gmm_workspace_floats(int M, int K, int D, int HW);

/* Same density when the context offsets are an embedding-table lookup (ContextEncoder(contexts,'embed','eyesample'), the only
 * form create_model builds: model.py:157,162): ctx_off[b] = cat_i tables[i][ctx[b,i]] (each row `width` wide, n_ctx*width =
 * 2*M*K*D).  The library buckets the batch by context tuple and hoists every sigma-dependent term per distinct scale
 * context, so no transcendental is evaluated per Gaussian.  n_ctx <= 2 and prod(cards) <= 2048, else CFPP_ERR_UNSUPPORTED
 * (use cfpp_embed_lookup + cfpp_gmm_logprob).  cards: HOST array; tables: HOST array of device pointers. */
int cfpp_gmm_logprob_ctxtab(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* wG,
                            const int64_t* ctx, int n_ctx, const int* cards, const float* const* tables, int width,
                            const float* logp_c, float logp_scale, float* out, void* workspace, int64_t workspace_bytes,
                            int B, int M, int K, int D, int HW, void* stream);
/* The same call for a caller that keeps `workspace` alive per parameter version: tables_ready != 0 says the parameter-only tables at its head
 * (1 / (2 sigma^2) and the log-normalisers per scale context) were filled by an earlier call with the same parameters, B and workspace. */
int cfpp_gmm_logprob_ctxtab_cached(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* wG,
                                   const int64_t* ctx, int n_ctx, const int* cards, const float* const* tables, int width,
                                   const float* logp_c, float logp_scale, float* out, void* workspace, int64_t workspace_bytes,
                                   int tables_ready, int B, int M, int K, int D, int HW, void* stream);
/* bytes of scratch for cfpp_gmm_logprob_ctxtab, or -1 when that context structure is unsupported */
int64_t cfpp_gmm_ctxtab_workspace_bytes(int B, int M, int K, int D, int HW, int n_ctx, const int* cards);

/* The same density as a register-tiled contraction (csrc/gmm_tile.cu): a tile of 64 samples x all M*K components per CTA, x and an
 * interleaved (mu, 1/(2 sigma^2)) table streamed through shared memory.  Two calls:
 *   cfpp_gmm_tile_prepare : builds the table (a function of the parameters only -- cache it per parameter version);
 *                           scale_table (n_scale_ctx, scale_width) optional: sigma = softplus(sG[m,k,e] + scale_table[v][scale_off + (m*K+k)*D + d])
 *                           gives one table per distinct scale context v (NULL: n_scale_ctx = 1, no offsets);
 *   cfpp_gmm_tile_logprob : ctx (B, n_ctx) int64 with n_ctx in {0, 1, 2} and cards (HOST) their cardinalities.  The batch is bucketed by
 *                           context tuple so that a tile shares one scale context (the LAST feature: the table must have cards[n_ctx-1]
 *                           scale contexts) and one mean-offset row mean_table[ctx[b,0]][mean_off + (m*K+k)*D + d] (mean_table NULL: none).
 * For ContextEncoder(contexts,'embed','eyesample') ('b (p m k d)', model.py:157,162): n_ctx == 2 -> means = tables[0], scales = tables[1],
 * offsets 0; n_ctx == 1 -> both from tables[0]: mean_off 0, scale_off M*K*D.  n_keys = product of cards (<= 4096).
 * M*K <= 128 (padded to a multiple of 4), K <= 64.  *_bytes return -1 when unsupported.
 * When M*K > 48 and x rows can be read as 16-byte vectors (x, x_bstride 16-byte aligned, D*HW a multiple of 4), cfpp_gmm_tile_logprob evaluates
 * the density on the tensor cores (csrc/gmm_tc.cu: tiles of 128 samples, tf32 hi/lo operands, K = 2 D*HW); a slice of a tile whose
 * parameters fail that kernel's accuracy guard, and every other x, takes the register-tiled kernel.  Both are deterministic. */
int64_t cfpp_gmm_tile_table_bytes(int M, int K, int D, int HW, int n_scale_ctx);
int cfpp_gmm_tile_prepare(const float* mG, const float* sG, const float* wG, const float* scale_table, int scale_width,
                          int scale_off, int n_scale_ctx, void* table, int M, int K, int D, int HW, void* stream);
int64_t cfpp_gmm_tile_workspace_bytes(int B, int M, int K, int D, int HW, int n_keys);
int cfpp_gmm_tile_logprob(const float* x, int64_t x_bstride, const void* table, const int64_t* ctx, int n_ctx, const int* cards,
                          const float* mean_table, int mean_width, int mean_off, const float* logp_c, float logp_scale,
                          float* out, void* workspace, int64_t workspace_bytes, int B, int M, int K, int D, int HW, void* stream);

/* ---- context encoders -------------------------------------------------------------------------------------- */
#define CFPP_MAX_CTX 8
#define CFPP_ENC_MAXC 64
enum { CFPP_EMB_ONEHOT = 0, CFPP_EMB_EYE = 1, CFPP_EMB_EMBED = 2, CFPP_EMB_DENSE = 3 /* embedding given as a (B,C) float matrix */ };
enum { CFPP_ENC_EYESAMPLE = 0, CFPP_ENC_UNIFORM = 1, CFPP_ENC_VARDEQ = 2, CFPP_ENC_ARGMAX = 3, CFPP_ENC_PROBSAMPLE = 4 };
/* ContextEncoder = Sequential(embedding, surjection) (model.py:30-90): context (B,n) int64 -> c (B,C), logp_c (B).
 * Embeddings: layers/rtdl/nn/_embeddings.py:103-109,140-150,265-283.  Surjections: layers/dequantize.py:55-63 (uniform),
 * :107-116 (variational), :239-268 (argmax bits, MSB first), :133-136 (eye), :152-161 (prob).  Inner flow:
 * FlowInvSequential.sample (layers/flowsequential.py:60-69) over ConditionalGaussianDistribution.sample
 * (distributions/gaussian.py:263-270) and 2 x [FC, ActNormFC, CouplingFC]. */
typedef struct {
  int emb, type, n_ctx, C;
  int card[CFPP_MAX_CTX];
  int bits[CFPP_MAX_CTX];
  int emb_dim;                              /* embed: columns per feature */
  const float* emb_w[CFPP_MAX_CTX];         /* embed: (card_i, emb_dim) */
  const float* dense;                       /* CFPP_EMB_DENSE: (B,C) already-embedded input */
  const float* qbins;                       /* (n_in) uniform/vardeq */
  const float* ldj_per_dim;                 /* (n_in) */
  const float* temperature;                 /* (1) sigmoid flow */
  int inner_dim;                            /* columns per feature of the inner (mean, log-scale) embedding = 2C/n_ctx */
  const float* inner_w[CFPP_MAX_CTX];       /* (card_i, inner_dim) */
  const float* fc[2];                       /* FC.NN (C,C) */
  const float* fc_logabsdet[2];             /* device scalars */
  const float* an_t[2];
  const float* an_logs[2];
  const float* cw1t[2]; const float* cb1[2];   /* CouplingFC: (C/2 -> 2C) packed K-major */
  const float* cw2t[2]; const float* cb2[2];   /* (2C -> 2C) */
  const float* cw3t[2]; const float* cb3[2];   /* (2C -> C) */
} cfpp_enc_desc;
/* noise: randn (B,C) for vardeq/argmax/probsample, rand (B,n_in) for uniform, NULL for eyesample.
 * emit_stage: -1 = full encoder; 0 / 1 = stop before ActNormFC #0 / #1 and write that (B,C) activation to c
 * (used once for the data-dependent ActNorm initialisation, layers/actnorm.py:53); 2 = stop after the conditional
 * Gaussian draw and write (x, log q) -- ConditionalGaussianDistribution.sample alone (gaussian.py:263-270). */
int cfpp_ctx_encode(const int64_t* ctx, const float* noise, float* c, float* logp_c, const cfpp_enc_desc* desc,
                    int emit_stage, int B, void* stream);
/* Several independent encoders over the same context batch in one launch (every specialist layer owns its own encoder:
 * 36 per forward for the CIFAR / ATM stacks).  descs_device: DEVICE array of n_enc descriptors (validated by the caller with
 * the same rules as cfpp_ctx_encode); noise / c_out / logp_out: HOST arrays of n_enc device pointers. */
#define CFPP_MAX_ENC_BATCH 64
int cfpp_ctx_encode_batch(const int64_t* ctx, const cfpp_enc_desc* descs_device, int n_enc, const float* const* noise,
                          float* const* c_out, float* const* logp_out, int B, void* stream);
/* The same launch for encoders that all carry the inner flow (type vardeq / argmax / probsample) and share one width C with a tiled
 * kernel (cfpp_ctx_encode_flow_supported(C) == 1: C = 8 -- eye + argmax over 68 ATM contexts --, C = 20 -- onehot [15, 5] + vardeq, the
 * CIFAR-10C stack): 128 samples of one encoder per CTA, the flow's parameters staged in shared memory, layer inputs in registers
 * (model.py:30-90, flowsequential.py:60-69, conv1x1.py:80-96, actnorm.py:86-102, coupling.py:80-97).  Same results as
 * cfpp_ctx_encode_batch up to fp32 summation order. */
int cfpp_ctx_encode_flow_supported(int C);
int cfpp_ctx_encode_batch_flow(const int64_t* ctx, const cfpp_enc_desc* descs_device, int n_enc, int C, const float* const* noise,
                               float* const* c_out, float* const* logp_out, int B, void* stream);
/* CatEmbeddings.forward (stack=False), layers/rtdl/nn/_embeddings.py:265-283: out[b] = cat_i tables[i][ctx[b,i]], each `width` wide.
 * `tables` is a HOST array of n_ctx device pointers. */
int cfpp_embed_lookup(const int64_t* ctx, const float* const* tables, int n_ctx, int width, float* out, int B, void* stream);
/* y (B,N) = act(x (B,K) @ wt (K,N) + b): the CN context networks (nn.Linear; coupling.py:37, actnorm.py:21, conv1x1.py:22). */
int cfpp_linear_fwd(const float* x, const float* wt, const float* b, float* y, int B, int K, int N, int relu, void* stream);
/* Every CN context network of a forward in ONE launch (coupling.py:37,45: Linear-ReLU-Linear-ReLU-Linear on the encoded context;
 * actnorm.py:21,44: Linear(C, 2D); conv1x1.py:22,32: Linear(C, D*D)).  Job j maps in[j] (B, K) through its chain of 1..3 linear
 * layers (ReLU between layers, none after the last) into out[j] (B, N[n_layers-1]).  Weights are K-major (K_l, N_l), K_0 = K,
 * K_l = N[l-1].  tril_dim = D > 0 declares the last layer's output a row-major (D, D) matrix of which the consumer reads only the
 * lower triangle and the diagonal (Conv1x1: tril(c,-1) + diag(exp(diag c)), conv1x1.py:36-40): the strictly upper entries are
 * neither computed nor written.  `jobs`, `in`, `out` are HOST arrays (n_jobs entries) of device pointers. */
#define CFPP_MAX_CN_JOBS 64
#define CFPP_CN_MAX_WIDTH 1024      /* K and hidden widths (everything staged in shared memory); the last N is unbounded */
typedef struct cfpp_cn_job {
  const float* w[3];
  const float* b[3];                /* (N_l) or NULL */
  int n_layers, K;
  int N[3];
  int tril_dim;
} cfpp_cn_job;
int cfpp_cn_batch(const cfpp_cn_job* jobs, int n_jobs, const float* const* in, float* const* out, int B, void* stream);


/* MaskedCoupling.forward (`--coupling maf`, layers/ar.py:35-57) after its masked residual block: h (B, 2C, HW) is the block's conv
 * output WITHOUT the identity; t = h[:, :C] + x, r = h[:, C:] + x (masked_conv_2d.py:92,98); z = x * exp(2 tanh(r/2)) + t;
 * ldj[b] = sum 2 tanh(r/2).  The block itself = three cfpp_conv2d_fwd launches (ReLU on the input) over mask-multiplied weights. */
/* y = max(x, 0): the pre-activation of MaskedResidualBlock2d (masked_conv_2d.py:94) in front of cfpp_conv_cond_tc_fwd. */
int cfpp_relu_fwd(const float* x, float* y, int64_t n, void* stream);
int cfpp_maf_coupling_fwd(const float* x, const float* h, float* z, float* ldj, int B, int C, int HW, void* stream);
/* the same for a --contextflow specialist (ar.py:39-42): h += add[b] ((B, 2C), broadcast over the pixels; may be NULL),
 * ldj[b] += logp_scale * logp_c[b] (logp_c may be NULL) */
int cfpp_maf_coupling_ctx_fwd(const float* x, const float* h, const float* add, const float* logp_c, float logp_scale,
                              float* z, float* ldj, int B, int C, int HW, void* stream);

/* Its backward: dh (B, 2C, HW) = cat(dz, dr), dr = (dz x s + dldj[b]) (1 - tanh^2(r/2)); dx = dz s + dz + dr (the identity feeds both halves);
 * the masked block's own input gradient is then accumulated onto dx by cfpp_conv2d_bwd_data(act = x, accumulate = 1). */
int cfpp_maf_coupling_bwd(const float* x, const float* h, const float* dz, const float* dldj, float* dx, float* dh,
                          int B, int C, int HW, void* stream);

/* ---- inverse (sampling) direction: SURVEY §8(f)-3 ------------------------------------------------------------ */
/* Coupling.reverse / TransCoupling.reverse, layers/coupling.py:68-73,150-155: t, r from h (+ add) as in cfpp_coupling_fwd;
 * x = cat(z[:, :C/2], (z[:, C/2:] - t) / exp(2 tanh(r/2))).  One HBM pass, 12*C*HW bytes/sample. */
int cfpp_coupling_inv(const float* z, const float* h, const float* add, float* x, int B, int C, int HW, void* stream);
/* ActNorm.reverse without context, layers/actnorm.py:73-78: x = z * exp(logs[d]) + t[d]. */
int cfpp_actnorm_inv(const float* z, float* x, const float* t, const float* logs, int B, int D, int HW, void* stream);
/* torch.inverse(NN), layers/conv1x1.py:70 (Conv1x1.reverse = cfpp_conv1x1_fwd with this matrix): fp64 Gauss-Jordan with
 * partial pivoting, D <= 128; singular[0] (optional, device int) = 1 when a zero pivot was met. */
int cfpp_mat_inverse(const float* A, int D, float* Ainv, int* singular, void* stream);
/* LogitTransform.reverse (layers/transforms.py:14-15): y = sigmoid(x). */
int cfpp_sigmoid_fwd(const float* x, float* y, int64_t n, void* stream);
/* Normalization.reverse (scalar scale), layers/normalize.py:37-41: x = (y - translation) * scale. */
int cfpp_normalize_inv(const float* y, float* x, int64_t n, float scale, float translation, void* stream);
/* Dequantization.reverse, layers/dequantize.py:19-20: y = floor(x). */
int cfpp_floor_fwd(const float* x, float* y, int64_t n, void* stream);
/* The image prologue backwards in one pass (model.py:97-100 right to left): Augment.reverse (keep the first C of C+A channels,
 * layers/augment.py:20-23), sigmoid, (v - t1) * s1, (v - t0) * s0, floor (do_floor).  x_cont (optional) = value before the floor. */
int cfpp_prologue_inv(const float* z, float* x, float* x_cont, int B, int C, int A, int HW,
                      float s1, float t1, float s0, float t0, int do_floor, void* stream);
/* GaussianMixtureDistribution.sample after its random draws (layers/distributions/gaussian.py:163-166: mixture m = 1 of
 * MixtureSameFamily(Categorical(softmax wG), Normal(mG, softplus sG))): x[b] = mG[m, comp[b]] + softplus(sG[m, comp[b]]) * eps[b];
 * comp (B) int64 component draws, eps (B, n_per_sample) standard-normal draws. */
int cfpp_gmm_sample(const float* mG, const float* sG, const int64_t* comp, const float* eps, float* x,
                    int B, int M, int K, int n_per_sample, int m, void* stream);

/* ---- loss / score epilogue: SURVEY §8(f)-2 ------------------------------------------------------------------- */
/* experiment_ad.py:204-211,262-281 / experiment_cl.py:127-133,185-204 after model.log_prob, in two launches:
 *   scaled (B,M) = dim_inv * logp with NaN -> 0;  lse (B) = logsumexp_m;  softmax1 (B) = softmax(scaled)[:,1] (1 when M = 1);
 *   last (B) = scaled[:, -1];  argmax (B) int64 (first maximum);
 *   sums[0] = sum_b logsigmoid(lse_b), sums[1] = sum_{b,m} logsigmoid(scaled), sums[2], sums[3] = numerator, denominator of
 *   nn.CrossEntropyLoss(weight=class_w)(scaled, gt) when gt != NULL (class_w NULL = unit weights).
 * cost_uns = -alpha * sums[0] / B (criterion) or -alpha * sums[1] / (B*M) (none); cost_sup = sums[2] / sums[3].
 * Every output but sums is optional (NULL).  Deterministic (fixed-order reductions, no atomics).
 * workspace: cfpp_score_workspace_bytes(B) device bytes. */
int64_t cfpp_score_workspace_bytes(int B);
int cfpp_score_epilogue(const float* logp, float dim_inv, const int64_t* gt, const float* class_w,
                        float* scaled, float* lse, float* softmax1, float* last, int64_t* argmax, float* sums,
                        void* workspace, int B, int M, void* stream);

/* ---- training direction, context-free conv stack: SURVEY §8(f)-1 ------------------------------------------------- */
/* What torch autograd derives for the reference (experiment_ad.py:204-213).  All gradients fp32; weight gradients are OVERWRITTEN;
 * every reduction over the batch has a fixed order (bit-identical run to run).
 * Coupling backward (layers/coupling.py:50-66): given x, h of the forward, dz and dldj (B, may be NULL):
 *   dx = cat(dz0, dz1 * s); dh = cat(dz1, (dz1 * x1 * s + dldj[b]) * (1 - tanh^2(r/2))), s = exp(2 tanh(r/2)), r = h_r (+ add_r: the
 *   additive context term `add` (B,C) of coupling.py:45, NULL without; its gradient is the sum of dh over the pixels: cfpp_rowsum).
 *   The conditioner's own gradient is then ADDED onto dx[:, :C/2] by cfpp_conv2d_bwd_data(accumulate = 1). */
int cfpp_coupling_bwd(const float* x, const float* h, const float* add, const float* dz, const float* dldj, float* dx, float* dh,
                      int B, int C, int HW, void* stream);
/* Context-conditioned (specialist) Conv1x1 / ActNorm, backward w.r.t. the input and the raw context-network output c
 * (layers/conv1x1.py:31-50, layers/actnorm.py:42-58; the frozen generalist parameters get no gradient under --contextflow).
 * Conv1x1: c (B,D,D): dx = W_b^T dz; dc = lower triangle of dz x^T, diagonal exp(c_ii) (dz x^T)_ii + HW dldj[b], zero above.
 * ActNorm: c (B,2D) 'b (p d)', base_t / base_logs (D) or NULL (conventional): dx = dz exp(-logs_b); dc = [-sum dz exp(-logs_b) |
 * -sum dz z + dldj[b]].  dx may be NULL. */
int cfpp_conv1x1_ctx_bwd(const float* x, const float* dz, const float* c, const float* NN, int contextflow, const float* dldj,
                         float* dx, float* dc, int B, int D, int HW, void* stream);
int cfpp_actnorm_ctx_bwd(const float* x, const float* dz, const float* c, const float* base_t, const float* base_logs,
                         const float* dldj, float* dx, float* dc, int B, int D, int HW, void* stream);
/* ActNorm backward without context (layers/actnorm.py:50-60): dx = dz * exp(-logs) (dx may be NULL);
 * dt[d] = -sum dz * exp(-logs); dlogs[d] = -sum dz * z + sum_b dldj[b].  workspace: cfpp_actnorm_bwd_workspace_floats(B, D) floats. */
int64_t cfpp_actnorm_bwd_workspace_floats(int B, int D);
int cfpp_actnorm_bwd(const float* x, const float* dz, const float* dldj, const float* t, const float* logs,
                     float* dx, float* dt, float* dlogs, float* workspace, int B, int D, int HW, void* stream);
/* One convolution of the conditioner (layers/coupling.py:26-29) with saved output, "same" reflect padding, torch weight layout
 * (Cout, Cin, KH, KW), KH, KW in {1, 3}: out = [relu](W * [relu](in) + bias); `relu` bit 0 = ReLU on the output, bit 1 = ReLU on the
 * input (the pre-activation order of MaskedResidualBlock2d, layers/autoregressive/masked_conv_2d.py:93-98).  `in` is read through a
 * batch stride (x0 is x[:, :C/2]). */
int cfpp_conv2d_fwd(const float* in, int64_t in_bstride, const float* W, const float* bias, float* out,
                    int B, int Cin, int Cout, int H, int Wd, int KH, int KW, int relu, void* stream);
/* din (= or +=, `accumulate`) the gradient of that convolution w.r.t. its input, including the adjoint of the reflect padding,
 * times (act > 0) when `act` (the input activation, post-ReLU) is given. */
int cfpp_conv2d_bwd_data(const float* dout, const float* W, const float* act, int64_t act_bstride, float* din, int64_t din_bstride,
                         int accumulate, int B, int Cin, int Cout, int H, int Wd, int KH, int KW, void* stream);
/* dW (Cout, Cin, KH, KW) and db (Cout, may be NULL) of that convolution.  With 1x1 kernels and Cin = Cout = D this is also
 * Conv1x1's dNN = sum_{b,p} dz x^T (layers/conv1x1.py:52-55).  Per-chunk partial sums go to `workspace`
 * (cfpp_conv2d_bwd_weight_workspace_floats floats) and are added in chunk order: deterministic, no atomics. */
int64_t cfpp_conv2d_bwd_weight_workspace_floats(int B, int Cin, int Cout, int KH, int KW);
int cfpp_conv2d_bwd_weight(const float* in, int64_t in_bstride, const float* dout, float* dW, float* db, float* workspace,
                           int B, int Cin, int Cout, int H, int Wd, int KH, int KW, void* stream);
/* g[i] = 0 where act[i] <= 0 (ReLU backward on a saved post-activation). */
int cfpp_relu_mask(float* g, const float* act, int64_t n, void* stream);
/* Conv1x1's log-det term: dNN[i][j] += HW * (sum_b dldj[b]) * inv[j][i], inv = cfpp_mat_inverse(NN). */
int cfpp_logdet_grad(float* dNN, const float* inv, const float* dldj, int B, int D, int HW, void* stream);
/* out[b] = sum_m g[b,m]: what a (B,) / (B,1) ldj term receives from the (B,M) accumulation (layers/flowsequential.py:23). */
int cfpp_rowsum(const float* g, float* out, int B, int M, void* stream);
/* Mixture base in training mode (layers/distributions/gaussian.py:142-161, context-free), M*K <= 256, n = D*H*W:
 *   prep: inv_var (M,K,n) = 1/softplus(sG)^2, cst (M,K) = log_softmax(wG) - sum log sigma - n/2 log 2pi;
 *   fwd : logp (B,M), resp (B,M,K) = component responsibilities (saved for the backward);
 *   bwd : given g = dL/dlogp (B,M): dx (B,n; may be NULL), dmG, dsG (M,K,n), dwG (M,K).
 *   workspace: cfpp_gmm_train_bwd_workspace_floats floats. */
int cfpp_gmm_train_prep(const float* sG, const float* wG, float* inv_var, float* cst, int M, int K, int n, void* stream);
int cfpp_gmm_train_fwd(const float* x, int64_t x_bstride, const float* mG, const float* inv_var, const float* cst,
                       float* logp, float* resp, int B, int M, int K, int n, void* stream);
int64_t cfpp_gmm_train_bwd_workspace_floats(int B, int M, int K, int n);
int cfpp_gmm_train_bwd(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* wG, const float* inv_var,
                       const float* resp, const float* g, float* dx, int64_t dx_bstride, float* dmG, float* dsG, float* dwG,
                       float* workspace, int B, int M, int K, int n, void* stream);

/* Mixture with per-sample context offsets (layers/distributions/gaussian.py:146-155), training direction: c (B, 2*M*K*D) 'b (p m k d)'
 * is the materialised context_net output (mean offsets | pre-softplus scale offsets).  fwd: logp (B,M) and the responsibilities resp
 * (B,M,K); bwd: dx (B, D*HW; may be NULL) and dc (B, 2*M*K*D).  The frozen mG / sG / wG get no gradient under --contextflow. */
int cfpp_gmm_ctx_train_fwd(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* wG, const float* c,
                           float* logp, float* resp, int B, int M, int K, int D, int HW, void* stream);
int cfpp_gmm_ctx_train_bwd(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* c, const float* resp,
                           const float* g, float* dx, int64_t dx_bstride, float* dc, int B, int M, int K, int D, int HW, void* stream);
/* Encoder flows in training mode: the base draw of ConditionalGaussianDistribution.sample (gaussian.py:263-270; c = [mean | log_scale]
 * (B, 2C), eps (B, C) standard normal: x = mean + exp(ls) eps, logq = sum(-1/2 log 2pi - ls - 1/2 eps^2)) and the epilogue of
 * VariationalCatDequantization.forward (dequantize.py:107-116: z = (xcat + sigmoid(u)) / qbins, ldj = ldj_const + sum(-softplus(-u) -
 * softplus(u)) - qu), each with the backward torch autograd derives.  The inner flow between them (FC, ActNormFC, CouplingFC) runs on
 * the Conv1x1 / ActNorm / Coupling training kernels with H = W = 1. */
int cfpp_cond_gauss_fwd(const float* c, const float* eps, float* x, float* logq, int B, int C, void* stream);
int cfpp_cond_gauss_bwd(const float* c, const float* eps, const float* dx, const float* dlogq, float* dc, int B, int C, void* stream);
/* mode 0: the vardeq form above; mode 1: ArgmaxCatDequantization (dequantize.py:239-268): z = sigmoid(u) * sign with sign = +-1 passed
 * in xcat, ldj = act - qu; mode 2: ProbSampling (:152-160): z = sigmoid(u), ldj = act + qu. */
int cfpp_vardeq_fwd(const float* u, const float* qu, const int64_t* xcat, const float* qbins, float ldj_const, int mode, float* z, float* ldj,
                    int B, int C, void* stream);
int cfpp_vardeq_bwd(const float* u, const int64_t* xcat, const float* qbins, int mode, const float* dz, const float* dldj, float* du, float* dqu,
                    int B, int C, void* stream);
/* Gradient of an embedding table (rtdl CatEmbeddings, _embeddings.py:265-283): dtable[v] = sum of dc[b, col0:col0+width] over the
 * samples b whose context feature equals v; perm (B) = sample indices stably sorted by that feature, offsets (cardinality + 1) the
 * bucket boundaries -- a fixed summation order, deterministic. */
int cfpp_embed_scatter(const float* dc, int64_t dc_stride, int col0, const int64_t* perm, const int64_t* offsets, float* dtable,
                       int cardinality, int width, void* stream);

/* ---- training direction of the SimpleViT conditioner (layers/simple_vit.py:30-127): SURVEY §8(f)-1 --------------------- */
/* Row-major token rows X (R = B * n_tok, F features).  Each entry is one op of the reference's module stack, forward with the
 * activations its backward needs, and the backward torch autograd would derive.  Reductions over rows are deterministic.
 * patchify: 'b c (h p1) (w p2) -> (b h w) (p1 p2 c)' (simple_vit.py:102); x read through a batch stride.  _inv: the inverse
 * permutation (the un-patchify of TransCoupling / the adjoint of patchify), stored or accumulated through a batch stride. */
int cfpp_patchify_fwd(const float* x, int64_t x_bstride, float* tok, int B, int c, int H, int W, int p1, int p2, void* stream);
int cfpp_patchify_inv(const float* tok, float* x, int64_t x_bstride, int accumulate, int B, int c, int H, int W, int p1, int p2, void* stream);
/* nn.LayerNorm(F) (eps 1e-5, biased variance): y, and mean / rstd per row for the backward.  F <= 320. */
int cfpp_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* rstd, int64_t R, int F, void* stream);
int64_t cfpp_layernorm_bwd_workspace_floats(int64_t R, int F);
int cfpp_layernorm_bwd(const float* x, const float* dy, const float* gamma, const float* mean, const float* rstd,
                       float* dx, float* dgamma, float* dbeta, float* workspace, int64_t R, int F, void* stream);
/* nn.Linear(I -> J): y = x W^T (+ bias), W (J, I) torch layout; its input gradient dx = dy W (stored or accumulated); dW = dy^T x, db. */
int cfpp_rows_linear_fwd(const float* x, const float* W, const float* bias, float* y, int64_t R, int I, int J, void* stream);
int cfpp_rows_linear_bwd_data(const float* dy, const float* W, float* dx, int accumulate, int64_t R, int I, int J, void* stream);
int64_t cfpp_rows_linear_bwd_weight_workspace_floats(int64_t R, int I, int J);
int cfpp_rows_linear_bwd_weight(const float* x, const float* dy, float* dW, float* db, float* workspace, int64_t R, int I, int J, void* stream);
/* nn.GELU() (erf form) and its derivative on the saved pre-activation. */
int cfpp_gelu_fwd(const float* x, float* y, int64_t n, void* stream);
int cfpp_gelu_bwd(const float* x, const float* dy, float* dx, int64_t n, void* stream);
/* x[r] += pos[r mod n_tok]  (the sincos position table, simple_vit.py:121). */
int cfpp_add_pos(float* x, const float* pos, int64_t R, int n_tok, int F, void* stream);
/* Single-head attention per sample (simple_vit.py:45-60, heads = 1, dim_head = 64): qkv rows (n_tok, 192) = [q | k | v];
 * P (B, n, n) = softmax(q k^T / 8) is saved; O = P v.  bwd: dqkv from dO. */
int cfpp_attention_fwd(const float* qkv, float* O, float* P, int B, int n_tok, void* stream);
int cfpp_attention_bwd(const float* qkv, const float* P, const float* dO, float* dqkv, int B, int n_tok, void* stream);

/* ---- rows beside the headline path (SURVEY 8f) ------------------------------------------------------------------- */
/* Standalone invertible activations on rows of D values (reference layers/activations.py:228-264).  kind 0 = Sigmoid(temperature):
 * z = sigmoid(T x), ldj[row] = sum_i log T - softplus(-T x_i) - softplus(T x_i); kind 1 = Softplus: z = softplus(x), ldj[row] = sum_i
 * logsigmoid(x_i).  inv: Sigmoid clamps z to [eps, 1 - eps] (the [0,1] assertion of :241 is the caller's), x = (log z - log1p(-z)) / T;
 * Softplus x = z + log1p(-exp(-max(z, eps))).  bwd: dx from dz (may be NULL) and dldj (rows; may be NULL).  temperature: device scalar. */
int cfpp_activation_fwd(const float* x, float* z, float* ldj, const float* temperature, int64_t rows, int D, int kind, void* stream);
int cfpp_activation_inv(const float* z, float* x, const float* temperature, int64_t n, float eps, int kind, void* stream);
int cfpp_activation_bwd(const float* x, const float* dz, const float* dldj, float* dx, const float* temperature, int64_t rows, int D,
                        int kind, void* stream);
/* StudentMixtureDistribution.log_prob (layers/distributions/student.py:44-111): logp (B, M) = Gaussian-mixture log-density + Student-t
 * mixture log-density of x (B, n = D*H*W) under parameters (M, K, n) / weights (M, K) (softmax over dim 0, renormalised along K by
 * Categorical).  prep fills `table` (cfpp_student_table_floats floats) from the parameters; redo it when they change. */
int64_t cfpp_student_table_floats(int M, int K, int n);
int cfpp_student_prep(const float* mG, const float* sG, const float* wG, const float* mS, const float* sS, const float* wS,
                      const float* vS, float* table, int M, int K, int n, void* stream);
int cfpp_student_logprob(const float* x, const float* table, float* logp, int B, int M, int K, int n, void* stream);
/* Training direction (vS frozen, as in the reference).  train_fwd: logp as above and resp (B, M, 2, K) = softmax_k of the Gaussian (0)
 * and Student-t (1) component terms, x rows at x_bstride floats.  train_bwd: from g (B, M) = dL/dlogp, dx (rows at dx_bstride; NULL
 * skips it) and, unless dmG is NULL, dmG, dsG, dmS, dsS (M, K, n) and dwG, dwS (M, K).  sG, wG, sS, wS are the raw parameters; table is
 * the one train_fwd read.  M*K <= 768.  Parameter sums run over fixed chunks of samples, then in chunk order: no atomics. */
int cfpp_student_train_fwd(const float* x, int64_t x_bstride, const float* table, float* logp, float* resp, int B, int M, int K, int n,
                           void* stream);
int64_t cfpp_student_train_bwd_workspace_floats(int B, int M, int K, int n);
int cfpp_student_train_bwd(const float* x, int64_t x_bstride, const float* table, const float* sG, const float* wG, const float* sS,
                           const float* wS, const float* resp, const float* g, float* dx, int64_t dx_bstride, float* dmG, float* dsG,
                           float* dwG, float* dmS, float* dsS, float* dwS, float* workspace, int B, int M, int K, int n, void* stream);
/* Training of the conventional (concatenated-context, contextflow = False) specialists.
 * bias_rows_relu: a (B, C, HW) <- relu(a + bias[b, c]) in place: conv1 of coupling.py:47 = W1[:, :D] x0 + (b1 + W1[:, D:] CN(c)).
 * gmm_ctx_param_bwd: gradients of the mixture's own mG, sG (M, K, D, HW) and wG (M, K) when they train beside the context offsets c
 * (B, 2*M*K*D) (distributions/gaussian.py:131-155); resp (B, M, K) from cfpp_gmm_ctx_train_fwd, g (B, M) = dL/dlogp. */
int cfpp_bias_rows_relu(float* a, const float* bias, int B, int C, int HW, void* stream);
int cfpp_gmm_ctx_param_bwd(const float* x, int64_t x_bstride, const float* mG, const float* sG, const float* wG, const float* c,
                           const float* resp, const float* g, float* dmG, float* dsG, float* dwG, int B, int M, int K, int D, int HW,
                           void* stream);

/* Fused multi-tensor AdamW (torch.optim.AdamW's update rule, model.py:289), capturable in a CUDA graph.  tensors: device array of
 * 4 pointers per tensor {param, grad, exp_avg, exp_avg_sq} (float32); chunks: device array of {tensor index, first element, count}
 * triples, count <= cfpp_adamw_chunk(); state: device float[3] {step count, 1 - b1^t, sqrt(1 - b2^t)} -- the call increments the
 * step count first; lr: device scalar.  Hyper-parameters arrive as doubles: 1 - beta and the bias corrections are formed in double, as
 * torch forms them from python floats, before rounding to float32. */
int cfpp_adamw_chunk(void);
int cfpp_adamw_step(const void* tensors, const int* chunks, int n_chunks, float* state, const float* lr, double beta1, double beta2,
                    double eps, double weight_decay, void* stream);

/* ---- container ------------------------------------------------------------------------------------------------ */
/* FlowSequential.forward, layers/flowsequential.py:23: logdet (B,M) += ldj (B,cols) with cols = 1 (broadcast) or M. */
int cfpp_ldj_accumulate(float* logdet, const float* ldj, int B, int M, int cols, void* stream);
/* The same accumulation for up to CFPP_LDJ_SUM_MAX terms in one launch, in the same order (bit-identical to the chain of
 * cfpp_ldj_accumulate calls): out (B,M) = [last +] (((first | 0) + terms[0]) + terms[1]) + ...; terms[k] is (B,cols[k]),
 * cols[k] in {1, M}; first / last optional (B,M) (flowsequential.py:20-27: logdet = 0 + sum ldj; logprob + logdet).
 * terms / cols: HOST arrays. */
#define CFPP_LDJ_SUM_MAX 64
int cfpp_ldj_sum(float* out, const float* first, const float* last, const float* const* terms, const int* cols, int n,
                 int B, int M, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CFPP_H_ */
