/*
 * virtex_b200 -- C ABI of the B200-native (sm_100a) kernels behind the VirTex bicaptioning pretraining step.
 *
 * The reference (kdexd/virtex) has no FFI of its own: its hot path is `VirTexModel.forward` + autograd
 * (virtex/models/captioning.py:71-143) executed by torch / torchvision library calls (SURVEY.md section 8b).
 * Each entry point below replaces one family of those library calls; the file:line it stands in for is cited.
 *
 * Conventions
 *   - plain pointers + sizes, no torch types; every pointer is a DEVICE pointer unless stated otherwise
 *   - `stream` is a cudaStream_t passed as void*
 *   - returns 0 on success, a negative VTX_E* code on failure; vtx_last_error() gives a message (thread local)
 *   - no allocation, no synchronisation, no global state beyond cached device properties
 *   - activations are bf16 (NHWC for the backbone, [tokens, features] row-major for the head); statistics,
 *     master parameters, gradients and the decoder residual stream are fp32
 */
#ifndef VIRTEX_B200_H_
#define VIRTEX_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VTX_OK 0
#define VTX_EINVAL (-1)
#define VTX_ECUDA (-2)
#define VTX_EUNSUPPORTED (-3)

const char* vtx_last_error(void);
int vtx_version(void);
/* Number of SMs of the current device (cached). */
int vtx_num_sms(void);

/* ------------------------------------------------------------------------------------------------------------------
 * tcgen05 GEMM:  D[M,N] = epilogue( sum_k A[m,k] * B[n,k] )       bf16 x bf16 -> fp32 accumulate in TMEM
 * Replaces every cuBLASLt / cuDNN GEMM-shaped call on the path: nn.Linear fwd/dgrad/wgrad
 * (virtex/modules/textual_heads.py:168-170,199,245,277; torch/nn/modules/transformer.py:1158-1199) and the 1x1 /
 * im2col'd convolutions of torchvision Bottleneck (torchvision/models/resnet.py:146-158).
 *   a_mn = 0: A is stored [M, K] row major (K contiguous, leading dim lda)     ("K-major")
 *   a_mn = 1: A is stored [K, M] row major (M contiguous, leading dim lda)     ("MN-major", used by wgrad)
 *   b_mn = 0: B is stored [N, K] row major;   b_mn = 1: B is stored [K, N] row major.
 * Epilogue order: acc -> (stats: per-column sum / sum of squares of acc, fp32 atomics) -> *alpha -> +bias[n]
 *                 -> +residual[m,n] (bf16) -> activation -> store (bf16 or fp32; or fp32 atomic accumulate).
 * split_k > 1 requires atomic = 1 (fp32 output, caller zero-initialises).
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct VtxGemm {
  const void* A;
  const void* B;
  void* D;
  const float* bias;    /* [N] or NULL */
  const void* residual; /* bf16 [M, ldr] or NULL */
  float* stats;         /* [2, N]: sum, sumsq  or NULL */
  int64_t lda, ldb, ldd, ldr;
  int32_t M, N, K;
  int32_t a_mn, b_mn;
  int32_t out_f32; /* 0: bf16 output, 1: fp32 output */
  int32_t atomic;  /* 1: D += result with fp32 atomics (needs out_f32) */
  int32_t act;     /* 0 none, 1 relu, 2 gelu(erf) */
  int32_t split_k; /* >= 1 */
  int32_t tile_n;  /* 0 = auto; else multiple of 16 (64 if b_mn) and <= 256 */
  float alpha;
  /* implicit 3x3 / stride 1 / pad 1 convolution over an NHWC bf16 tensor (conv_c > 0):
     A is the activation [conv_n, conv_h, conv_w, conv_c]; M = n*h*w, K = 9*conv_c, B = weights [N, (kh,kw,c)].
     conv_wgrad = 1 swaps roles for the weight gradient (see gemm_tc.cu). */
  int32_t conv_n, conv_h, conv_w, conv_c;
  int32_t conv_mode; /* 0 = plain GEMM, 1 = implicit fprop/dgrad gather on A (64->64 channel problems run the halo-reuse
                        variant automatically), 2 = wgrad gather on B,
                        4 = halo-reuse wgrad for C = Cout = 64: A = dy, B = x, D[9*C, Cout] fp32 += (atomic),
                            i.e. the TRANSPOSE of mode 2's [Cout, 9*C] output,
                        5 = 7x7/2 stem fprop over the space-to-depth view S written by vtx_stem_s2d: A = S
                            [conv_n, conv_h + 3, conv_w + 3, 16] (conv_h x conv_w = OUTPUT size, conv_c = 64 = 4 pixels
                            x 16 channels), B = packed weights [64, 256] (vtx_stem_s2d_w_pack), D [n*h*w, 64] NHWC
                            (torchvision resnet.py:197 conv1 forward, BN statistics through `stats`),
                        6 = stem wgrad: A = dy [conv_n, conv_h, conv_w, 64], B = S; D [64, 256] fp32 += (atomic) */
  int32_t conv_stride;          /* conv_mode 1 / 2 only: 0 or 1 = unit stride; 2 = stride-2 convolution -- conv_h / conv_w
                                   are the INPUT extent, outputs (M, K of the wgrad) run over (h-1)/2+1 x (w-1)/2+1; the
                                   gather uses TMA traversal strides (torchvision resnet.py:133-138, 239-243) */
  int32_t conv_taps;            /* 0 or 9 = 3x3 / pad 1 taps; 1 = a single tap (1x1 / pad 0: the strided downsample) */
  /* conv_mode 1, explicit tap grid (conv_taps_h > 0): conv_taps_h x conv_taps_w taps, tap (a, b) reads (h + a - conv_pad,
     w + b - conv_pad); K = taps * conv_c.  With the output view below this is one parity class of a stride-2 dgrad. */
  int32_t conv_taps_h, conv_taps_w, conv_pad;
  /* conv_mode 1, output view (conv_out_w > 0): D is the strided sub-grid [conv_n, conv_out_h, conv_out_w, N] of a larger
     NHWC tensor with element strides ldd_n / ldd_h / ldd_w (D points at its first element); rows of the conv_h x conv_w
     tile grid that fall outside the view are clipped. */
  int32_t conv_out_h, conv_out_w;
  int64_t ldd_w, ldd_h, ldd_n;
  const uint8_t* residual_mask; /* optional (plain bf16 GEMMs, N % 32 == 0): bit (m, n) of a [M, N/8] bit mask in the layout
                                   vtx_bn_act writes; residual[m, n] is added only where the bit is set.  This is the
                                   shortcut gradient dz = dOut * [block output > 0] of a bottleneck without dz ever being
                                   written to memory (torchvision resnet.py:160-161 backward). */
  /* BatchNorm-backward reduction fused into the epilogue (bnr_y != NULL; bf16 output, N % 8 == 0, no bias / activation /
     stats): D is the gradient w.r.t. the output of a train-mode BN (+ReLU) whose pre-BN input is bnr_y (same geometry as
     D: leading dimension bnr_ldy, or D's view strides for conv_mode 1 output views) and whose forward parameters are
     bnr_bnp [4, N] = mean, invstd, scale, shift (vtx_bn_finalize).  With dz = D * mask, mask = bit (m, n) of bnr_mask
     (layout of vtx_bn_act's mask, plain GEMMs only) or, when bnr_mask is NULL, [bnr_y * scale + shift > 0],
         bnr_sums[0, n] += sum_m dz[m, n],    bnr_sums[1, n] += sum_m dz[m, n] * (bnr_y[m, n] - mean[n]) * invstd[n]
     -- exactly what vtx_bn_bwd_reduce computes in a separate pass over D and y (torch batch_norm backward, first half);
     D itself is stored unmasked, vtx_bn_bwd_finalize_apply consumes the sums. */
  const void* bnr_y;
  const float* bnr_bnp;
  float* bnr_sums;
  const uint8_t* bnr_mask;
  int64_t bnr_ldy;
} VtxGemm;

int vtx_gemm(const VtxGemm* g, void* stream);
/* Tile schedule of the persistent GEMM.  0 (default): static round robin, tile t of CTA c = c + i * #CTAs -- the fastest
   when the GEMM has the GPU to itself.  1: every CTA takes its tiles from a per-launch atomic counter, so that an SM held
   by another stream's kernel (NCCL's all-reduce CTAs during the overlapped gradient exchange of the data-parallel step,
   scripts/pretrain_virtex.py:121-123) does not own a fixed share of every GEMM issued meanwhile.  Process-wide. */
int vtx_gemm_set_dynamic_schedule(int on);
/* sizeof(VtxGemm) of the built library (a binding compares it with its own struct definition) */
int vtx_sizeof_gemm(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Backbone auxiliaries (NHWC bf16 activations).  Replace cuDNN BatchNorm / ATen elementwise + pooling kernels called by
 * torchvision/models/resnet.py:143-163,268-276 and the im2col side of strided convolutions.
 * ------------------------------------------------------------------------------------------------------------------ */
/* 7x7/stride 2/pad 3 stem: image fp32 NCHW -> cols bf16 [N*Ho*Wo, ldc], k = (kh*7+kw)*3 + c, zero padded to ldc */
int vtx_stem_im2col(const float* img, void* cols, int N, int H, int W, int ldc, void* stream);
/* space-to-depth view of the image for the 4-tap implicit stem conv (vtx_gemm conv_mode 5 / 6):
   image fp32 NCHW [N, 3, H, W] -> S bf16 [N, H/2 + 3, W/2 + 3, 16],
   S[n, i, j, (r*2+q)*3 + c] = img[n, c, 2i + r - 3, 2j + q - 3], zero outside the image and in channels 12..15 */
int vtx_stem_s2d(const float* img, void* S, int N, int H, int W, void* stream);
/* conv1.weight fp32 [O, 3, 7, 7] -> bf16 [O, 256], k = a*64 + b*16 + (r*2+q)*3 + c for tap (kh, kw) = (2a+r, 2b+q) */
int vtx_stem_s2d_w_pack(const float* w, void* wp, int O, void* stream);
/* grad fp32 [O, 3, 7, 7] += dwp fp32 [O, 256] (same index map) */
int vtx_stem_s2d_w_unpack_add(const float* dwp, float* grad, int O, void* stream);
/* 3x3 / pad 1 / given stride: x [N,H,W,C] -> cols [N*Ho*Wo, 9*C] (k = tap*C + c) and its adjoint */
int vtx_im2col3x3(const void* x, void* cols, int N, int H, int W, int C, int stride, void* stream);
int vtx_col2im3x3(const void* dcols, void* dx, int N, int H, int W, int C, int stride, void* stream);
/* strided 1x1 (downsample) gather and its adjoint (dx += scatter(dxs)) */
int vtx_subsample(const void* x, void* xs, int N, int H, int W, int C, int stride, void* stream);
int vtx_upsample_add(const void* dxs, void* dx, int N, int H, int W, int C, int stride, void* stream);
/* stats [2,C] (sum, sumsq from the GEMM epilogue) -> bnp [4,C] = mean, invstd, scale, shift; updates running stats */
int vtx_bn_finalize(const float* stats, float count, const float* gamma, const float* beta, float* running_mean,
                    float* running_var, int64_t* num_batches_tracked, float momentum, float eps, int training,
                    float* bnp, int C, void* stream);
/* out = act(y*scale + shift [+ res | + res*scale_r + shift_r]).  relu_mask (optional, relu only): uint8 [M, C/8], bit j
   of byte (m, g) = [pre-activation of channel 8g + j > 0] -- all that BN backward needs of `out` (1/16 of its bytes) */
int vtx_bn_act(const void* y, const float* bnp, const void* res, const float* bnp_res, void* out, uint8_t* relu_mask,
               int64_t M, int C, int relu, void* stream);
/* vtx_bn_finalize + vtx_bn_act fused into one launch */
int vtx_bn_finalize_act(const float* stats, float count, const float* gamma, const float* beta, float* running_mean,
                        float* running_var, int64_t* num_batches_tracked, float momentum, float eps, int training,
                        float* bnp, const void* y, const void* res, const float* bnp_res, void* out, uint8_t* relu_mask,
                        int64_t M, int C, int relu, void* stream);
int vtx_bn_relu_maxpool(const void* y, const float* bnp, void* out, uint8_t* idx, int N, int H, int W, int C,
                        void* stream);
int vtx_maxpool_bwd(const void* dpool, const uint8_t* idx, void* da, int N, int H, int W, int C, void* stream);
/* BN backward in three steps: per-channel sums of dz and dz*xhat (dz = dA*[relu_mask bit]); coefficients + dgamma/dbeta;
   dy = scale*(dz - mean(dz) - xhat*mean(dz*xhat)).  A second BN sharing dz (downsample branch) rides along.
   relu_mask: the uint8 bit mask written by vtx_bn_act / vtx_bn_finalize_act, or NULL;
   relu_mask == NULL && mask_from_y: the ReLU mask is recomputed as [y*scale + shift > 0] instead of being read. */
int vtx_bn_bwd_reduce(const void* dA, const uint8_t* relu_mask, const void* y, const float* bnp, const void* y2,
                      const float* bnp2, float* sums, float* sums2, int64_t M, int C, int mask_from_y,
                      void* stream);
int vtx_bn_bwd_finalize(const float* sums, const float* bnp, float count, float* coef, float* dgamma, float* dbeta,
                        int C, void* stream);
int vtx_bn_bwd_apply(const void* dA, const uint8_t* relu_mask, const void* y, const float* bnp, const float* coef, void* dy,
                     const void* y2, const float* bnp2, const float* coef2, void* dy2, void* dz_out, int64_t M, int C,
                     int mask_from_y, void* stream);
/* vtx_bn_bwd_finalize + vtx_bn_bwd_apply fused into one launch (dgamma/dbeta accumulated by the first thread block) */
int vtx_bn_bwd_finalize_apply(const float* sums, const float* sums2, float count, float* dgamma, float* dbeta,
                              float* dgamma2, float* dbeta2, const void* dA, const uint8_t* relu_mask, const void* y,
                              const float* bnp, void* dy, const void* y2, const float* bnp2, void* dy2, void* dz_out,
                              int64_t M, int C, int mask_from_y, void* stream);
/* conv weight layouts: fp32 OIHW <-> bf16 [O, (kh,kw,I)] GEMM operand; flipped/transposed dgrad operand */
int vtx_conv_w_pack(const float* w, void* out, int O, int I, int KH, int KW, int ldk, void* stream);
int vtx_conv_w_pack_dgrad(const float* w, void* out, int O, int I, void* stream);
int vtx_conv_w_unpack_add(const float* dwp, float* grad, int O, int I, int KH, int KW, int ldk, void* stream);
/* same for the transposed [(tap, I), O] weight-gradient layout written by vtx_gemm conv_mode 4 */
int vtx_conv_w_unpack_add_t(const float* dwt, float* grad, int O, int I, int KH, int KW, void* stream);
/* Batched form of the six weight-layout kernels above (and of vtx_stem_s2d_w_pack / _unpack_add): one launch executes a
   DEVICE-resident table of jobs.  kind: 0 pack, 1 pack_dgrad, 2 unpack_add, 3 unpack_add_t, 4 stem s2d pack,
   5 stem s2d unpack_add, 6 pack for parity class (KH, KW) of a stride-2 3x3 dgrad ([I, taps*O], see backbone.cu), 7 transpose of a 1x1 weight ([O, I] -> bf16 [I, O]); total = number of output elements of the job; block0 = first thread block of the job (jobs are
   sorted by block0, every block handles vtx_weight_job_block_elems() consecutive elements). */
typedef struct VtxWeightJob {
  const void* src;
  void* dst;
  int64_t total;
  int32_t O, I, KH, KW, ldk, kind, block0, reserved;
} VtxWeightJob;
int vtx_conv_w_jobs(const VtxWeightJob* jobs, int njobs, int total_blocks, void* stream);
int vtx_weight_job_block_elems(void);
int vtx_cast_bf16(const float* in, void* out, int64_t n, void* stream);
int vtx_nhwc_to_nchw_f32(const void* in, float* out, int N, int HW, int C, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Textual-head auxiliaries.  `seed` is a DEVICE pointer to the 64-bit dropout seed of the current step (so a captured
 * CUDA graph can be replayed with fresh masks); `site` distinguishes dropout call sites; p = 0 disables dropout.
 * Replace nn.Embedding/LayerNorm/Dropout (virtex/modules/embedding.py:58-73), F.scaled_dot_product_attention with
 * the merged float mask (torch/nn/functional.py:6608-6682), GELU, nn.CrossEntropyLoss (virtex/models/captioning.py:69).
 * ------------------------------------------------------------------------------------------------------------------ */
int vtx_embed_fwd(const int64_t* tokens, const float* words, const float* positions, const float* gamma,
                  const float* beta, float* z, float* stats, float* out, void* out_bf, int M, int T, int H, int pad,
                  float eps, float p, const uint64_t* seed, uint32_t site, void* stream);
int vtx_embed_bwd(const float* dy_a, const void* dy_b, const int64_t* tokens, const float* z, const float* stats,
                  const float* gamma, float* d_words, float* d_pos, float* d_gamma, float* d_beta, int M, int T, int H,
                  int pad, float p, const uint64_t* seed, uint32_t site, void* stream);
/* z = res + dropout(branch); out = LN(z) (ln=1) or z (ln=0) */
int vtx_add_ln_fwd(const float* res, const void* branch, const float* gamma, const float* beta, float* z, float* stats,
                   float* out, void* out_bf, int M, int H, float eps, float p, const uint64_t* seed, uint32_t site,
                   int ln, void* stream);
int vtx_ln_bwd(const float* dy_a, const void* dy_b, const float* z, const float* stats, const float* gamma,
               const float* d_skip, float* d_res, void* d_branch, float* d_gamma, float* d_beta, int M, int H, float p,
               const uint64_t* seed, uint32_t site, int ln, void* stream);
/* attention core, head_dim 64, Tq <= 32, Tk <= 64; causal = 1: key j visible to query i iff j <= i and j < lengths[b];
   causal = 2: iff j < lengths[b] (key-padding mask only: masked language modelling); causal = 0: every key */
int vtx_attn_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* out,
                 int64_t ldo, float* lse, int B, int heads, int Tq, int Tk, const int64_t* lengths, int causal,
                 float p, const uint64_t* seed, uint32_t site, void* stream);
int vtx_attn_bwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const void* dout,
                 int64_t ldo, const float* lse, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv,
                 int B, int heads, int Tq, int Tk, const int64_t* lengths, int causal, float p, const uint64_t* seed,
                 uint32_t site, void* stream);
int vtx_gelu_dropout_fwd(const void* u, void* h, int64_t n, float p, const uint64_t* seed, uint32_t site, void* stream);
int vtx_gelu_dropout_bwd(const void* dh, const void* u, void* du, int64_t n, float p, const uint64_t* seed,
                         uint32_t site, void* stream);
/* shift = 1: the target of position t is tokens[b, t+1] (captioning.py:111-114); shift = 0: tokens[b, t] is the label of
   position t itself (masked_labels of virtex/models/masked_lm.py:68-72).  Targets equal to pad are ignored. */
int vtx_count_valid(const int64_t* tokens, int B, int T, int pad, int shift, float* count, void* stream);
/* logits bf16 [B*T, ldl]; loss += mean NLL over valid targets; write_grad: logits := dlogits in place */
int vtx_cross_entropy(void* logits, int64_t ldl, const int64_t* tokens, int B, int T, int V, int pad, int shift,
                      const float* count, float* loss, int write_grad, void* stream);
int vtx_colsum(const void* X, int64_t ld, int M, int N, float* out, void* stream);
int vtx_argmax_rows(const float* X, int64_t ld, int M, int N, int64_t* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Beam-search decoding (csrc/decode.cu).  Replace the per-step full-prefix recomputation of
 * virtex/models/captioning.py:165-213 (decoding_step: visual features repeated per beam, the textual head over every
 * position) and the selection / history arithmetic of virtex/utils/beam_search.py (AutoRegressiveBeamSearch.search).
 * ------------------------------------------------------------------------------------------------------------------ */
/* Single-query attention, head_dim 64, one query per (row, head): out[r, h] = softmax_j(q . k_j / 8) v_j over Tk keys.
   Key / value j of row r start at k / v + phys * row_stride + j * pos_stride (+ h * 64), elements:
     table == NULL: phys = r / group (cross attention: group = rows per image, keys = the image's visual tokens);
     table != NULL: phys = table[r * ldt + j] for j < Tk - 1 and r for the newest key j = Tk - 1 (self attention over
                    a position-major KV cache whose history rows are reordered by vtx_beam_reorder, never moved).
   Tk <= cache_len <= 64, heads * 64 % 128 == 0. */
int vtx_decode_attn(const void* q, int64_t ldq, const void* k, const void* v, int64_t row_stride, int64_t pos_stride,
                    const int32_t* table, int ldt, int group, void* out, int64_t ldo, int rows, int heads, int Tk,
                    int cache_len, void* stream);
/* One beam-search selection over fp32 logits [images * beam_in, ldl] (beam_search.py search loop body): one block per
   row, one thread-block cluster per image.  Per row: lp = log_softmax; lp[last token] = -10000; a row whose last token
   is eos scores 0 at eos and -inf elsewhere (its logits are not read); top per_node of the row, each plus the row's
   running score.  Per image: top beam_out of the beam_in * per_node candidates.  Order everywhere: NaN above every
   number (as in vtx_argmax_rows), then larger, then lower token id within a row / lower (beam, rank) candidate index
   within an image.  Outputs [images * beam_out]: tokens, parents (the selected candidate's ROW index,
   image * beam_in + beam), scores.  last == NULL: first step (no penalty, no forcing, running scores 0; beam_in = 1,
   per_node = beam_out).  ended (optional) := nonzero iff every selected token is eos.
   per_node <= min(16, V), beam_in <= 8. */
int vtx_beam_step(const float* logits, int64_t ldl, int V, int images, int beam_in, int per_node, int beam_out,
                  int eos, const int64_t* last, const float* scores_in, int64_t* tokens, int64_t* parents,
                  float* scores_out, int32_t* ended, void* stream);
/* Follow the parents of a beam step: out_hist[r, :n_hist] = in_hist[parents[r], :n_hist], out_hist[r, n_hist] = tokens[r]
   (int64 [rows, ldh]); with out_table, the cache index of vtx_decode_attn for n_tab cached positions:
   out_table[r, j] = in_table[parents[r], j] for j < n_tab - 1, out_table[r, n_tab - 1] = parents[r] (int32 [rows, ldt]).
   Not in place. */
int vtx_beam_reorder(const int64_t* parents, const int64_t* tokens, const int64_t* in_hist, int64_t* out_hist, int ldh,
                     int n_hist, const int32_t* in_table, int32_t* out_table, int ldt, int n_tab, int rows,
                     void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Classification pretext heads (csrc/classify.cu).  Replace the global average pooling of LinearTextualHead
 * (virtex/modules/textual_heads.py:46-95), the per-image K-hot loss loop and the top-10 of
 * virtex/models/classification.py:69-107.  The linear layer between pooling and loss is a vtx_gemm.
 * ------------------------------------------------------------------------------------------------------------------ */
/* NHWC bf16 backbone output feat [B*S, C] -> pooled bf16 [B, C] = mean over the S positions of each image (fp32
   accumulation, one rounding).  S >= 1, C % 8 == 0, 16-byte aligned pointers. */
int vtx_avgpool_fwd(const void* feat, void* pooled, int B, int S, int C, void* stream);
/* dfeat bf16 [B*S, C] = dpooled fp32 [B, C] / S, broadcast over the S positions of each image. */
int vtx_avgpool_bwd(const float* dpooled, void* dfeat, int B, int S, int C, void* stream);
/* K-hot cross entropy over fp32 logits [B, ldl]: the label set of image b is the ids of labels int64 [B, L] inside
   [0, V), minus the ids of `ignore` [n_ignore] (duplicates count once; other ids are skipped, never dereferenced).
   loss[0] += sum_b (lse_b - mean_{v in set} z_bv) / B, NaN for an image whose set is empty.  dlogits != NULL: bf16
   [B, lddl] := (softmax - [v in set] / K) / B, a zero row where K = 0; columns >= V are not written.
   V <= 65536, L <= 1024, ldl % 4 == 0, lddl % 8 == 0. */
int vtx_khot_xent(const float* logits, int64_t ldl, const int64_t* labels, int L, const int64_t* ignore, int n_ignore,
                  int B, int V, float* loss, void* dlogits, int64_t lddl, void* stream);
/* out int64 [M, k] = indices of the k largest of each fp32 row X [M, ld] (first N columns), best first.  Order: NaN
   above every number, then larger value, then lower index (the rule of vtx_argmax_rows).  1 <= k <= min(16, N). */
int vtx_topk_rows(const float* X, int64_t ld, int M, int N, int k, int64_t* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * GPU input pipeline (csrc/input_pipe.cu): decoded uint8 HWC images -> fp32 NCHW network input, token lists -> padded
 * matrices.  Replaces the per-sample albumentations / cv2 transforms and the collate of
 * virtex/data/datasets/captioning.py:51-100 with the transform lists of virtex/factories.py:131-155.  Random parameters
 * are sampled on the host.  src: all images of the batch back to back (uint8, RGB, HWC), image n at src + src_off[n];
 * geom_i [B,8] = {H, W, region y0, x0, h, w, window offset y, x}; geom_d [B,2] = {region h / resized h, region w /
 * resized w}; jit_i [B,6] = {flip, apply-jitter, op order[4] (0 brightness, 1 contrast, 2 saturation, 3 hue)};
 * jit_d [B,4] = the four factors.  Integer paths are bit-exact with OpenCV's uint8 resize / cvtColor / addWeighted.
 * ------------------------------------------------------------------------------------------------------------------ */
/* crop + cv2.resize(INTER_LINEAR) (+ horizontal flip): out uint8 [B, S, S, 3] */
int vtx_image_resample(const uint8_t* src, const int64_t* src_off, const int32_t* geom_i, const double* geom_d,
                       const int32_t* jit_i, uint8_t* out, int B, int S, void* stream);
/* gray_sum[n] += sum of grey values of image n at the contrast stage of its jitter (caller zero-initialises) */
int vtx_image_gray_sum(const uint8_t* img, const int32_t* jit_i, const double* jit_d, uint64_t* gray_sum, int B, int S,
                       void* stream);
/* colour jitter in the sampled op order + (v - mean*255) / (std*255), written as fp32 NCHW; norm = {m[3], 1/s[3]} */
int vtx_image_jitter_normalize(const uint8_t* img, const int32_t* jit_i, const double* jit_d, const uint64_t* gray_sum,
                               const float* norm, float* out, int B, int S, void* stream);
/* flat token ids + offsets [B+1] -> caption / reversed caption [B, T] right-padded with pad, lengths [B] (<= max_len) */
int vtx_collate_tokens(const int64_t* flat, const int64_t* offs, int64_t* cap, int64_t* rev, int64_t* lengths, int B,
                       int T, int max_len, int64_t pad, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Fused optimiser tail over flat fp32 arenas (scripts/pretrain_virtex.py:157-162; virtex/factories.py:529-545;
 * virtex/optim/lookahead.py:82-102).  segs: device array of {int64 begin, int64 end, float lr, float wd}.
 * ctl[0] = gradient scale (clip / world size), ctl[1] = gradient norm; hyper = {lr multiplier, first step, lookahead}.
 * ------------------------------------------------------------------------------------------------------------------ */
int vtx_sumsq(const float* x, int64_t n, float* out, void* stream);
int vtx_clip_coef(const float* sumsq, int world_size, float max_norm, float* ctl, void* stream);
int vtx_sgd_step(float* p, const float* g, float* mom, float* slow, void* p_bf, const void* segs, int nseg,
                 const float* ctl, const float* hyper, float momentum, float la_alpha, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VIRTEX_B200_H_ */
