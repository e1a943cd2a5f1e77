/* omnidata_b200 — C ABI of the B200-native DPT-Hybrid-384 hot path.
 *
 * This header is the drop-in boundary (SURVEY.md §8b).  The reference (EPFL-VILAB/omnidata) is pure
 * Python/PyTorch on this path and has no FFI of its own; every entry point below replaces a chain
 * of torch library calls made by a reference function, cited as `file:line` under
 * omnidata_tools/torch/ (M/ = modules/midas/, L/ = losses/).  timm 0.4.12 (pinned by
 * requirements.txt:15, called at M/vit.py:483) is not vendored in the reference; its arithmetic
 * is cited as "timm <symbol>".
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name says host; no torch types cross this ABI;
 *   - activations are channels-last (NHWC / token-major) bf16 unless stated; strides are in
 *     ELEMENTS, the channel stride is always 1;
 *   - an `int32_t dtype` (or x_dtype / y_dtype) parameter is an odb_dtype naming the storage type of the
 *     activation tensors of that call (bf16 in production, fp32 in the correctness mode);
 *   - every function only enqueues work on `stream` (a cudaStream_t passed as void*); nothing
 *     allocates, synchronises or touches the host heap — safe under CUDA-graph capture;
 *   - return value: 0 on success, a negative odb_status otherwise; odb_last_error() returns a
 *     thread-local message.  There is NO CPU fallback: without a CUDA device every compute entry
 *     point fails with ODB_ERR_CUDA.
 */
#ifndef OMNIDATA_B200_H_
#define OMNIDATA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ODB_ABI_VERSION 4

typedef enum odb_status {
  ODB_OK = 0,
  ODB_ERR_INVALID = -1, /* bad argument / unsupported shape */
  ODB_ERR_CUDA = -2,    /* CUDA runtime or driver error (message has the detail) */
  ODB_ERR_UNSUPPORTED = -3
} odb_status;

typedef enum odb_act { ODB_ACT_NONE = 0, ODB_ACT_RELU = 1, ODB_ACT_GELU = 2 } odb_act;

/* Storage type of an activation tensor.  bf16 is the production format; fp32 carries the ViT residual stream
 * (the reference adds every block's output to an fp32 stream: timm Block.forward `x = x + ...`) and every
 * activation of the fp32 correctness mode (SURVEY.md 8c: the reference itself is fp32-only). */
typedef enum odb_dtype { ODB_DTYPE_BF16 = 0, ODB_DTYPE_F32 = 1 } odb_dtype;

/* A strided channels-last view [b][h][w][c] (bf16 storage unless the owning descriptor says fp32; strides in
 * elements of the storage type). */
typedef struct odb_view {
  const void* ptr;
  int32_t c, w, h, b;
  int64_t sx, sy, sb; /* element strides of w, h, b */
} odb_view;

#define ODB_MAX_VIEWS 4
#define ODB_MAX_TAPS 9

/* Implicit-GEMM convolution / linear layer on tcgen05 tensor cores:
 *
 *   out[b,y,x,n] = epilogue( sum_{t<num_taps} sum_{c<C} view[tap_view[t]][b, y+tap_dy[t], x+tap_dx[t], c]
 *                                                     * weight[n][t*C + c] )
 *
 * Reads outside a view are zero (TMA out-of-bounds fill) — this is the convolution padding.
 * A stride-2 convolution is expressed with up to four parity-plane views (doubled strides).
 * A linear layer is the degenerate case num_taps = 1, h = b = 1, w = rows.
 *
 * epilogue(v) = residual + act(v + bias)        (each term optional), stored as bf16 to `out`
 *               and, if out2.ptr != NULL, relu(.) of the same value to `out2`.
 *
 * Replaces, depending on the call site: nn.Linear in timm Attention/Mlp (loop M/vit.py:150-151),
 * timm HybridEmbed.proj (M/vit.py:133), ProjectReadout.project (M/vit.py:36-47),
 * act_postprocess convs (M/vit.py:431-462), scratch.layerN_rn (M/blocks.py:49-75, used
 * M/dpt_depth.py:73-76), ResidualConvUnit_custom.conv1/conv2 (M/blocks.py:263-286),
 * FeatureFusionBlock_custom.out_conv (M/blocks.py:339), output_conv[0] (M/dpt_depth.py:91),
 * timm ResNetV2 StdConv2dSame layers.
 */
typedef struct odb_conv_gemm_desc {
  int32_t num_views;
  odb_view views[ODB_MAX_VIEWS]; /* all views share c = C (multiple of 8; K blocks of 64) */
  int32_t num_taps;
  int8_t tap_view[ODB_MAX_TAPS];
  int8_t tap_dx[ODB_MAX_TAPS];
  int8_t tap_dy[ODB_MAX_TAPS];
  const void* weight; /* bf16 [n][num_taps * C], K contiguous */
  int32_t n;          /* output channels */
  odb_view out;       /* c = n; w,h,b = output extent */
  odb_view out2;      /* optional relu copy (ptr may be NULL) */
  const float* bias;  /* fp32 [n] or NULL */
  int64_t bias_sb;    /* 0, or n for a per-image bias [b][n] (ProjectReadout cls term) */
  odb_view residual;  /* optional bf16 residual, same extent as out (ptr may be NULL); sb may be 0 */
  int32_t act;        /* odb_act */
  int32_t tile_w, tile_h; /* spatial tile of the 128-row MMA tile, tile_w*tile_h <= 128; 0 = auto */
  int32_t block_n;        /* N tile: 256, 128, 64 (32 with the head tail); 0 = auto */
  int32_t cta_pair;       /* tcgen05 cta_group::2 (two SMs per 256-row tile): 0 = auto, 1 = on, -1 = off */
  int32_t halo;           /* 3x3 stride-1 pad-1 convs: load one halo tile per K block and address the nine
                           * taps inside it (3x less input traffic): 0 = auto (currently off: the deeper per-tap ring measured
                           * faster on every layer of this network), 1 = on, -1 = off */
  /* Fused DPT head tail (M/dpt_depth.py:93-97): only with n == 32.  When head_out != NULL the
   * 32-channel result relu(v + bias) is not stored; instead
   *   head_out[b][k][y][x] = relu?(head_b[k] + sum_j head_w[k][j] * relu(v_j + bias_j))  (fp32, NCHW) */
  const float* head_w; /* fp32 [head_c][32] */
  const float* head_b; /* fp32 [head_c] */
  int32_t head_c;
  int32_t head_relu;
  float* head_out;
  /* Fused GroupNorm statistics (timm GroupNormAct after every StdConv2dSame): when gn_partial != NULL
   * each epilogue warp also writes, for the rows it owns, the per-group (sum, sum of squares)
   * of its 32 rows to  gn_partial[b][ty*tiles_x+tx][quadrant 0..3][group][2]  (fp32, every entry is
   * written exactly once: no atomics, deterministic).  The sums are taken over the UNROUNDED fp32 accumulators
   * (timm GroupNormAct normalises the fp32 conv output), not over the stored bf16 values.  odb_groupnorm_finalize reduces them. */
  float* gn_partial;
  int32_t gn_groups;
  /* Epilogue code path: 0 = auto (a specialised straight-line epilogue — TMEM read of the next 64-column
   * chunk in flight, residual fetched by TMA into the output staging slot — whenever the flags are
   * bias[+relu|+gelu] or bias+residual with a plain strided residual; the generic epilogue otherwise),
   * -1 = always the generic epilogue.  Both produce bit-identical results. */
  int32_t epilogue;
  /* Storage types (odb_dtype).  in_dtype: views + weight.  out_dtype: out, out2, residual.
   *   (BF16, BF16)  the tcgen05 tensor-core path described above;
   *   (BF16, F32)   tensor-core path with an fp32 epilogue: out = residual + (acc + bias), residual and out fp32
   *                 (requires bias and residual, no act / out2 / gn / head): the ViT residual stream;
   *   (F32,  F32)   fp32 correctness mode: the same contraction on the FP32 FMA pipe (weight fp32 [n][taps*C]),
   *                 partial sums combined in fp64; bias / act / residual / out2 as above, no gn_partial / head. */
  int32_t in_dtype;
  int32_t out_dtype;
  /* Activation of the out2 copy: ODB_ACT_NONE / ODB_ACT_RELU = relu (ResidualConvUnit's `relu(out)` operand),
   * ODB_ACT_GELU = exact-erf GELU (train mode: out keeps the pre-activation of mlp.fc1 for the backward, out2 feeds fc2). */
  int32_t out2_act;
} odb_conv_gemm_desc;

int odb_conv_gemm(const odb_conv_gemm_desc* desc, void* stream);
/* The tiling odb_conv_gemm will use for `desc`: out4 = {tiles_x, tiles_y, block_n, flags}, flags bit 0 =
 * CTA pair, bit 1 = halo mode. */
int odb_conv_gemm_plan(const odb_conv_gemm_desc* desc, int32_t* out4);

/* LayerNorm over the last dim (timm Block.norm1/norm2, eps 1e-6): y = (x-mean)/sqrt(var+eps)*g + b.
 * x, y bf16 [rows][cols] (cols multiple of 256, <= 1024); gamma/beta fp32. */
int odb_layernorm(const void* x, const float* gamma, const float* beta, void* y, int64_t rows,
                  int32_t cols, float eps, int32_t x_dtype, int32_t y_dtype, void* stream);

/* Fused multi-head attention (timm Attention.forward): qkv bf16 [b][tokens][3][heads][64] as written
 * by the qkv linear; out bf16 [b][tokens][heads*64]; softmax(q k^T * scale) v.  tcgen05 kernel:
 * S and O accumulate in TMEM, exact two-pass fp32 softmax (global row maximum), P rounded to bf16
 * for the PV product, fp32 row sum of the unrounded P.  Up to 640 tokens all K / V blocks of an (image, head) stay
 * resident in shared memory; above 640 tokens a second kernel with the same arithmetic streams them through a ring
 * of shared-memory stages, one work unit per (image, head, 128-query tile).  lse (optional, training, tokens <= 640
 * only; ODB_ERR_UNSUPPORTED above): fp32 [b][heads][tokens] = log2 of the row's sum of exp2(s * scale * log2 e),
 * what odb_attention_bwd re-normalises with. */
int odb_attention(const void* qkv, void* out, float* lse, int32_t b, int32_t tokens, int32_t heads, float scale,
                  void* stream);
/* fp32 correctness mode of odb_attention: qkv fp32 [b][tokens][3][heads][64], out fp32 [b][tokens][heads*64];
 * dot products and the PV sum in fp64, exp / division exact (no fast-math).  Up to 640 tokens a score row is kept
 * in shared memory; above 640 tokens a kernel with no score buffer makes three passes over the keys (row maximum,
 * fp64 sum of exp(s - max), PV with s and exp recomputed), with the same definitions. */
int odb_attention_f32(const float* qkv, float* out, int32_t b, int32_t tokens, int32_t heads, float scale,
                      void* stream);

/* fp32 correctness mode of the DPT head tail (M/dpt_depth.py:95-97; the tensor-core path fuses this into
 * odb_conv_gemm's head epilogue): x fp32 [b][h][w][32] = relu(conv3x3 + bias), out[b][k][y][x] = relu?(bias[k] +
 * sum_j w[k][j] x[..j]) fp32 NCHW; `pre` (optional) receives the value before the final ReLU. */
int odb_head_tail_f32(const float* x, const float* w, const float* bias, float* out, float* pre, int32_t b,
                      int32_t h, int32_t wd, int32_t head_c, int32_t relu, void* stream);

/* GroupNorm statistics (timm GroupNormAct, 32 groups), deterministic (no floating-point atomics):
 * stats fp32 [b][groups][2] = (mean, 1/sqrt(var + eps)) over x bf16 [b][hw][c], biased variance,
 * reduced in a fixed order with fp64 combination.  `scratch` is caller-owned device memory of at
 * least odb_groupnorm_scratch_bytes(...) bytes, 256-byte aligned, ZEROED ONCE at allocation (the
 * kernel leaves it zeroed); it may be shared by successive calls on one stream. */
int64_t odb_groupnorm_scratch_bytes(int32_t b, int32_t hw, int32_t c, int32_t groups);
int odb_groupnorm_stats(const void* x, float* stats, void* scratch, int64_t scratch_bytes, int32_t b,
                        int32_t hw, int32_t c, int32_t groups, float eps, int32_t dtype, void* stream);

/* Reduce the partial sums written by odb_conv_gemm (gn_partial) in a fixed order with fp64
 * combination: stats[b][g] = (mean, 1/sqrt(var + eps)); rows_per_image = tiles_x * tiles_y * 4,
 * count = pixels * channels_per_group of one group. */
int odb_groupnorm_finalize(const float* partial, float* stats, int32_t b, int32_t rows_per_image,
                           int32_t groups, double count, float eps, void* stream);

/* GroupNorm apply (+ optional shortcut, + optional ReLU), timm Bottleneck.forward:
 *   y = relu?( gn(x; stats, gamma, beta) + shortcut )
 * shortcut = 0 (res == NULL) | res (res_stats == NULL) | gn(res; res_stats, res_gamma, res_beta). */
int odb_groupnorm_apply(const void* x, const float* stats, const float* gamma, const float* beta,
                        const void* res, const float* res_stats, const float* res_gamma,
                        const float* res_beta, void* y, int32_t b, int32_t hw, int32_t c,
                        int32_t groups, int32_t relu, int32_t dtype, void* stream);

/* Stem tail (timm ResNetV2 stem.norm + stem.pool): GroupNorm+ReLU then MaxPool 3x3 stride 2 with
 * TF-SAME padding (0,1).  x bf16 [b][h][w][c] -> y bf16 [b][h/2][w/2][c]. */
int odb_stem_gn_relu_maxpool(const void* x, const float* stats, const float* gamma,
                             const float* beta, void* y, int32_t b, int32_t h, int32_t w, int32_t c,
                             int32_t groups, int32_t dtype, void* stream);

/* im2col for the 7x7 stride-2 TF-SAME stem conv (timm StdConv2dSame 3->64): x fp32 NCHW
 * [b][3][h][w] -> cols bf16 [b*(h/2)*(w/2)][kpad], column (ky*7+kx)*3+ch, zero padded. */
int odb_stem_im2col(const float* x, void* cols, int32_t b, int32_t h, int32_t w, int32_t kpad,
                    int32_t dtype, void* stream);

/* Bilinear x2 upsampling, align_corners=True (M/blocks.py:335-337, M/dpt_depth.py:93), fused with
 * the skip add of the next fusion block (M/blocks.py:330): out = up2(z) + res; out_relu = relu(out).
 * z bf16 [b][h][w][c]; res/out/out_relu bf16 [b][2h][2w][c]; res and out_relu may be NULL. */
int odb_upsample2x_add(const void* z, const void* res, void* out, void* out_relu, int32_t b,
                       int32_t h, int32_t w, int32_t c, int32_t dtype, void* stream);

/* Patch embedding gather of the plain ViT backbones (DPT-Large `vitl16_384`, `vitb16_384`; timm PatchEmbed =
 * Conv2d(3, D, patch, stride patch), applied at M/vit.py:131): x fp32 NCHW [b][3][h][w] ->
 * cols bf16 [b * (h/patch) * (w/patch)][3 * patch * patch], column (c * patch + py) * patch + px = the row-major
 * flattening of the conv weight, so the embedding is one odb_conv_gemm. */
int odb_patchify(const float* x, void* cols, int32_t b, int32_t h, int32_t w, int32_t patch, int32_t dtype,
                 void* stream);

/* tokens[b][0][:] = cls + pos[0]  (M/vit.py:135-147); tokens bf16 [b][tokens][c]; cls, pos0 fp32 [c]. */
int odb_write_cls_row(void* tokens, const float* cls, const float* pos0, int32_t b, int32_t tokens_n,
                      int32_t c, int32_t dtype, void* stream);

/* ProjectReadout cls term (M/vit.py:43-47): out[b][n] = bias[n] + sum_k w[n][c + k] * tokens[b][0][k]
 * w bf16 [c][2c] (the Linear(2c, c) weight), tokens bf16 [b][tokens][c], out fp32 [b][c]. */
int odb_readout_cls_bias(const void* w, const float* bias, const void* tokens, float* out, int32_t b,
                         int32_t tokens_n, int32_t c, int32_t dtype, void* stream);

/* dst bf16[n] = round(src fp32[n]) (n a multiple of 8): the hooked ViT activations (M/vit.py:158-165 `get_activation`)
 * leave the fp32 residual stream as bf16 operands of the readout GEMM. */
int odb_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream);

/* =====================================================================================================
 * Backward of the network (train_depth.py:183-190 training_step -> loss.backward(); PL runs autograd over
 * the reference modules).  dgrad of every conv / linear layer is odb_conv_gemm itself with the re-packed
 * (in/out swapped, 180-degree rotated) weight from odb_pack_weight; the entry points below are the rest.
 * `dtype` is the storage type of activations and activation gradients; statistics, affine parameters,
 * parameter gradients and the ViT residual-stream gradient are fp32.  All reductions have a fixed order.
 * ===================================================================================================== */

/* Weight gradient of a convolution / linear layer described like odb_conv_gemm (views + taps):
 *   out[n][t * C + c] (+)= sum_{b,y,x} dy[b,y,x,n] * view[tap_view[t]][b, y + tap_dy[t], x + tap_dx[t], c]
 * i.e. the gradient in the PACKED weight layout of odb_conv_gemm (fp32).  bf16: tcgen05 kernel with both
 * operands MN-major straight from the channels-last tensors (the 128-byte-swizzled TMA box of 64 pixels x 64
 * channels that feeds the forward as a K-major A tile IS the MN-major operand of the transposed product),
 * split over the pixel range, fp32 partials in `workspace`, ordered reduction.  fp32: FP32-pipe twin. */
typedef struct odb_wgrad_desc {
  int32_t num_views;
  odb_view views[ODB_MAX_VIEWS];
  int32_t num_taps;
  int8_t tap_view[ODB_MAX_TAPS];
  int8_t tap_dx[ODB_MAX_TAPS];
  int8_t tap_dy[ODB_MAX_TAPS];
  odb_view dy;            /* c = n; w, h, b = the layer's output extent */
  int32_t n;
  float* out;             /* fp32 [n][num_taps * C] */
  void* workspace;        /* split partials */
  int64_t workspace_bytes;
  int32_t accumulate;     /* add to `out` instead of overwriting */
  int32_t dtype;          /* odb_dtype of views and dy */
} odb_wgrad_desc;
int64_t odb_conv_wgrad_workspace_bytes(const odb_wgrad_desc* desc);
int odb_conv_wgrad(const odb_wgrad_desc* desc, void* stream);

/* Backward of odb_attention (timm Attention.forward): dqkv [b][tokens][3][heads][64] from qkv, the forward output o
 * [b][tokens][heads*64], its gradient d_o, and (bf16 path) the per-row log2-sum-exp `lse` fp32 [b][heads][tokens]
 * that odb_attention wrote.  bf16: P and dS are re-materialised per (image, head) by tcgen05 GEMMs with fused
 * softmax / dS epilogues, dQ / dK / dV are three more batched GEMMs; fp32: FP32-pipe twin (lse unused). */
int64_t odb_attention_bwd_workspace_bytes(int32_t b, int32_t tokens, int32_t heads, int32_t dtype);
int odb_attention_bwd(const void* qkv, const void* o, const void* d_o, const float* lse, void* dqkv, void* workspace,
                      int64_t workspace_bytes, int32_t b, int32_t tokens, int32_t heads, float scale, int32_t dtype,
                      void* stream);

/* out = a + b * [mask > 0]   (a, mask optional): ReLU backward and gradient accumulation; n elements (multiple of 8). */
int odb_mask_add(const void* a, const void* b, const void* mask, void* out, int64_t n, int32_t dtype, void* stream);
/* exact-erf GELU (nn.GELU() default) forward on a stored pre-activation, and its backward du = dy * gelu'(u). */
int odb_gelu_fwd(const void* u, void* y, int64_t n, int32_t dtype, void* stream);
int odb_gelu_bwd(const void* dy, const void* u, void* du, int64_t n, int32_t dtype, void* stream);
/* Bias gradients: out[bt][n] (+)= sum over rows of x[bt][row][n] (row / batch strides in elements). */
int64_t odb_colsum_workspace_bytes(int32_t batches, int64_t rows_per_batch, int32_t n);
int odb_colsum(const void* x, float* out, void* workspace, int32_t batches, int64_t rows_per_batch, int32_t n,
               int64_t row_stride, int64_t batch_stride, int32_t accumulate, int32_t dtype, void* stream);
/* out[bt][i] (+)= sum_p partial[bt][p][i] in fp64, in a fixed order (8 interleaved part lanes, then the lanes). */
int odb_reduce_partials(const float* partial, float* out, int32_t batches, int32_t parts, int64_t n, int32_t accumulate,
                        void* stream);
/* LayerNorm backward on the fp32 residual stream: ds_out = ds_in + dLN(dy; x, gamma) (ds_in may be NULL), optional
 * copy of ds_out in `dtype` (the next GEMM operand), dgamma / dbeta (+)=, and optionally (dcolsum != NULL) the column
 * sums of ds_out (+)= : the bias gradient of the linear layer whose output gradient ds_out is (timm Block: attn.proj
 * after norm2's backward, the previous block's mlp.fc2 after norm1's). */
int64_t odb_layernorm_bwd_workspace_bytes(int32_t cols);
int odb_layernorm_bwd(const void* dy, const float* x, const float* gamma, const float* ds_in, float* ds_out, void* ds_copy,
                      float* dgamma, float* dbeta, float* dcolsum, void* workspace, int64_t rows, int32_t cols, float eps,
                      int32_t accumulate, int32_t dtype, void* stream);
/* GroupNorm backward (timm GroupNormAct): g = dy * [mask > 0] (mask NULL: g = dy; the mask is the stored output of the
 * ReLU that follows the norm); dx, dgamma (+)=, dbeta (+)= from x and the forward statistics (mean, rstd). */
int64_t odb_groupnorm_bwd_workspace_bytes(int32_t b, int32_t hw, int32_t c, int32_t groups);
int odb_groupnorm_bwd(const void* dy, const void* mask, const void* x, const float* stats, const float* gamma, void* dx,
                      float* dgamma, float* dbeta, void* workspace, int32_t b, int32_t hw, int32_t c, int32_t groups,
                      int32_t accumulate, int32_t dtype, void* stream);
/* Adjoint of odb_upsample2x_add's bilinear part: dz [b][h][w][c] from dout [b][2h][2w][c]. */
int odb_upsample2x_bwd(const void* dout, void* dz, int32_t b, int32_t h, int32_t w, int32_t c, int32_t dtype, void* stream);
/* Backward of odb_stem_gn_relu_maxpool down to the GroupNorm output: g_s0 [b][h][w][c] = gradient w.r.t. gn(s0), already
 * masked by the ReLU; the pooling gradient goes to the first maximum of each window (torch semantics). */
int odb_stem_pool_bwd(const void* dt, const void* s0, const float* stats, const float* gamma, const float* beta, void* g_s0,
                      int32_t b, int32_t h, int32_t w, int32_t c, int32_t groups, int32_t dtype, void* stream);
/* DPT head tail, unfused (training): out[b][k][y][x] = relu?(bias[k] + sum_j w[k][j] a[b][y][x][j]), a has
 * channel_stride channels per pixel of which the first 32 are used; and its backward (da zero in the padding channels). */
int odb_head_tail_fwd(const void* a, int32_t channel_stride, const float* w, const float* bias, float* out, int32_t b,
                      int32_t h, int32_t wd, int32_t head_c, int32_t relu, int32_t dtype, void* stream);
int64_t odb_head_tail_bwd_workspace_bytes(int32_t head_c);
int odb_head_tail_bwd(const float* dout, const float* out, const void* a, int32_t channel_stride, const float* w, void* da,
                      float* dw, float* dbias, void* workspace, int32_t b, int32_t h, int32_t wd, int32_t head_c,
                      int32_t relu, int32_t accumulate, int32_t dtype, void* stream);
/* ds_out (fp32) = ds_in (fp32, optional) + g (`dtype`); optional copy of ds_out in `dtype`. */
int odb_add_cast(const float* ds_in, const void* g, float* ds_out, void* copy, int64_t n, int32_t dtype, void* stream);
/* train_depth.py:263 `torch.clamp(depth_preds, 0, 1)` and its backward: out = (g1 + g2) * [0 <= p <= 1] (g2 optional). */
int odb_clamp01(const float* p, float* out, int64_t n, void* stream);
int odb_clamp01_bwd(const float* p, const float* g1, const float* g2, float* out, int64_t n, void* stream);
/* Per-step weight packing: w fp32 [n][c][taps] (optionally weight-standardised, timm StdConv2dSame eps) ->
 * fwd `dtype` [n_pad][taps * c_pad] (odb_conv_gemm weight) and bwd `dtype` [c_pad][taps * n_pad] (dgrad weight). */
int odb_pack_weight(const float* w, void* fwd, void* bwd, int32_t n, int32_t c, int32_t taps, int32_t n_pad, int32_t c_pad,
                    int32_t standardize, float eps, int32_t dtype, void* stream);
/* Multi-tensor forms: one launch for a whole table of layers.  `items` is a DEVICE array of n_items records
 *   pack:   { const float* w; void* fwd; void* bwd; int32 n, c, taps, n_pad, c_pad, standardize, first_block, first_tile; }
 *   unpack: { const float* gp; const float* w; float* dw; int32 n, c, taps, c_pad, standardize, first_block, pad, pad; }
 * first_block / first_tile: prefix sums of n_pad (pack rows), ceil(n_pad/32)*ceil(c_pad/32)*taps (transpose tiles), n (unpack
 * rows); total_rows / total_tiles their totals; max_row_floats = max taps * c_pad over the table. */
int odb_pack_weights_multi(const void* items, int32_t n_items, int32_t total_rows, int32_t total_tiles, float eps, int32_t dtype,
                           void* stream);
int odb_unpack_wgrads_multi(const void* items, int32_t n_items, int32_t total_rows, int32_t max_row_floats, float eps,
                            void* stream);
/* Packed-layout weight gradient gp fp32 [n][taps * c_pad] -> parameter layout dw fp32 [n][c][taps], through the weight
 * standardisation when `standardize` (w = the fp32 parameter). */
int odb_unpack_wgrad(const float* gp, const float* w, float* dw, int32_t n, int32_t c, int32_t taps, int32_t c_pad,
                     int32_t standardize, float eps, void* stream);

/* ---- depth-training losses (train_depth.py:261-279), forward and (odb_*_bwd) backward with respect to the
 * prediction; all tensors fp32 [b][h][w] ------- */

/* make_valid_mask (train_depth.py:215-242): valid = nearest_upsample(max_pool2d(1 - mask, pool)) == 0. */
int odb_make_valid_mask(const float* mask_float, uint8_t* mask_valid, int32_t b, int32_t h, int32_t w,
                        int32_t pool, void* stream);

/* MidasLoss(alpha, scales, reduction='image-based').forward (losses/midas_loss.py:137-157):
 * out3 = (total, ssi, reg).  mask: uint8, 1 = valid.  Exact lower nanmedian by radix select,
 * deterministic fp64-combined reductions.  workspace: >= odb_midas_loss_workspace_bytes(b), 256-B aligned. */
int64_t odb_midas_loss_workspace_bytes(int32_t b);
int odb_midas_loss_fwd(const float* prediction, const float* target, const uint8_t* mask, int32_t b,
                       int32_t h, int32_t w, float alpha, int32_t scales, float* out3, void* workspace,
                       int64_t workspace_bytes, void* stream);

/* VNL_Loss.forward(first, second, select) (losses/virtual_normal_loss.py:151-194) for given point
 * triplets p1/p2/p3 (device int32 [n_points], flat index y*w + x — the reference draws them with host
 * NumPy RNG, :52-72).  `first` takes the reference's `gt_depth` slot (train_depth.py:272 passes the
 * PREDICTION there).  group_loss: scratch fp32 [b * n_points]; out1: the scalar loss. */
int odb_vnl_loss_fwd(const float* first, const float* second, const int32_t* p1, const int32_t* p2,
                     const int32_t* p3, int32_t n_points, int32_t b, int32_t h, int32_t w, float fx, float fy,
                     float delta_z, int32_t select, float* out1, float* group_loss, void* stream);

/* Backward of MidasLoss: grad[b][h][w] = d(w_ssi * ssi + w_reg * reg) / d(prediction) exactly as autograd derives it
 * for losses/midas_loss.py:137-157 (ssi through the median element and the deviation; reg through prediction_ssi AND
 * through the least-squares scale / shift).  Call after odb_midas_loss_fwd on the SAME prediction / target / mask with
 * its workspace untouched (fwd_workspace).  For train_depth.py:276 `ssi + 0.1 * reg`: w_ssi = 1, w_reg = 0.1.
 * bwd_workspace: odb_midas_loss_bwd_workspace_bytes(b) bytes; gbuf: scratch fp32 [b][h][w].  Deterministic. */
int64_t odb_midas_loss_bwd_workspace_bytes(int32_t b);
int odb_midas_loss_bwd(const float* prediction, const float* target, const uint8_t* mask, int32_t b, int32_t h,
                       int32_t w, int32_t scales, float w_ssi, float w_reg, const void* fwd_workspace,
                       void* bwd_workspace, float* gbuf, float* grad, void* stream);

/* Backward of VNL_Loss.forward(first, second) with respect to `first` (train_depth.py:272: the prediction):
 * grad fp32 [b][h][w] = upstream * d(loss)/d(first).  Call after odb_vnl_loss_fwd with the same arguments and its
 * group_loss untouched.  acc: scratch, 8 bytes per pixel (64-bit fixed-point accumulators: the scatter over points
 * sampled with replacement is bit-reproducible); sel4: scratch, 4 doubles. */
int odb_vnl_loss_bwd(const float* first, const float* second, const int32_t* p1, const int32_t* p2, const int32_t* p3,
                     int32_t n_points, int32_t b, int32_t h, int32_t w, float fx, float fy, int32_t select,
                     const float* group_loss, float upstream, void* acc, double* sel4, float* grad, void* stream);

/* Normal-training loss pair (SURVEY.md 8(f) rank 2; train_normal.py:247-258): with
 * preds = clamp(prediction, 0, 1) when clamp_prediction != 0,
 *   l1  = masked_l1_loss(preds, target, mask x3)                 (losses/masked_losses.py:4-7)
 *   cos = masked_cosine_angular_loss(preds, target, mask x3)      (losses/masked_losses.py:14-23)
 *   out3 = (cos + 10 * l1, l1, cos).
 * prediction, target fp32 [b][3][h][w]; mask_valid uint8 [b][h][w] (odb_make_valid_mask); workspace: 3 * b doubles.
 * Deterministic (fixed-order fp64 partial sums); backward: odb_normal_loss_bwd. */
int odb_normal_loss_fwd(const float* prediction, const float* target, const uint8_t* mask_valid, int32_t b,
                        int32_t h, int32_t w, int32_t clamp_prediction, float* out3, double* workspace,
                        void* stream);

/* ---- optimizer step of the depth train step (row a21: train_depth.py:381-383 Adam(lr), :425 gradient_clip_val=10)
 * over FLAT fp32 buffers holding all parameters / gradients / moments.
 *
 * odb_clip_grad_norm: torch.nn.utils.clip_grad_norm_(params, max_norm) without the host round trip:
 * out2 = (total L2 norm, clip coefficient min(1, max_norm / (norm + 1e-6))) on the device; the gradients are NOT
 * modified — odb_adam_step applies the coefficient while it reads them.  workspace: odb_grad_norm_workspace_bytes()
 * bytes, 256-byte aligned, zero-filled ONCE by the caller.  Deterministic (fixed-order fp64 partial sums).
 *
 * odb_adam_step: torch.optim.Adam update (betas, eps as given; no weight decay, no amsgrad), step = 1, 2, …;
 * clip2 = the out2 of odb_clip_grad_norm or NULL (no clipping).  step_scalars (device fp32 [2], may be NULL): when given,
 * the two step-dependent scalars (lr / (1 - beta1^step), sqrt(1 - beta2^step)) are read from device memory instead of
 * being computed from `step` — what a CUDA-graph replay of the train step needs; odb_adam_step_scalars (host function,
 * host pointer) computes them exactly as odb_adam_step does. */
int64_t odb_grad_norm_workspace_bytes(void);
int odb_clip_grad_norm(const float* grads, int64_t n, float max_norm, void* workspace, float* out2, void* stream);
int odb_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                  const float* clip2, float lr, float beta1, float beta2, float eps, int64_t step,
                  const float* step_scalars, void* stream);
int odb_adam_step_scalars(float lr, float beta1, float beta2, int64_t step, float* out2_host);

/* ---- 3-D refocus augmentation (SURVEY.md 8(f) rank 4; data/refocus_augmentation.py) ------------------------------
 * odb_refocus_quantiles: compute_quantiles (:82-87): quantile_vals fp32 [b][n_quantiles + 1] = torch.quantile(depth[b],
 * i / n_quantiles) (linear interpolation; exact order statistics by radix select), first -= eps, last += eps.
 * odb_refocus_compose: refocus_image (:144-157) after the blur radii are known: the Gaussian blur stack
 * (separable, replicate padding, cutoff int(3 r) made odd, r < 0.1 = copy; radii fp32 [b][levels]) and the per-pixel
 * blend of the two levels bracketing the pixel's depth with weights 1 - dist^2.  rgb fp32 [b][3][h][w], depth fp32
 * [b][h][w], out fp32 [b][3][h][w]; stack_tmp / stack: scratch fp32 [b][levels][3][h][w] each; segments (optional)
 * int32 [b][h][w] = the left quantile index (`return_segments`). */
int odb_refocus_quantiles(const float* depth, int32_t b, int32_t h, int32_t w, int32_t n_quantiles, float eps,
                          float* quantile_vals, void* stream);
int odb_refocus_compose(const float* rgb, const float* depth, const float* quantile_vals, const float* blur_radii,
                        int32_t b, int32_t h, int32_t w, int32_t levels, float* stack_tmp, float* stack, float* out,
                        int32_t* segments, void* stream);

/* Backward of the normal-training loss pair: grad fp32 [b][3][h][w] = d(w_l1 * l1 + w_cos * cos) / d(prediction)
 * (through the clamp when clamp_prediction != 0); for train_normal.py:258 `cos + 10 * l1`: w_l1 = 10, w_cos = 1.
 * fwd_workspace: the workspace odb_normal_loss_fwd filled for the same inputs. */
int odb_normal_loss_bwd(const float* prediction, const float* target, const uint8_t* mask_valid, int32_t b, int32_t h,
                        int32_t w, int32_t clamp_prediction, float w_l1, float w_cos, const double* fwd_workspace,
                        float* grad, void* stream);

int odb_fill_zero(void* ptr, int64_t bytes, void* stream);

/* ---- image pre- / post-processing either side of the forward (SURVEY.md 8(f) rank 1) ------------
 *
 * odb_pil_resize_crop_to_tensor replaces transforms.Resize(384, BILINEAR) + CenterCrop(384) + ToTensor
 * [+ Normalize(0.5, 0.5)] of omnidata_tools/torch/demo.py:74-76,92-95 for an 8-bit image already on the
 * device (src: uint8 [src_h][src_w][channels], channels 1 or 3, row pitch src_pitch bytes).  Pillow's
 * resize is an antialiased two-pass triangle filter in 8-bit fixed point (ImagingResample, 22 fractional
 * bits, 8-bit intermediate); the kernels evaluate exactly that, so `out` is bit-identical to the
 * reference's input tensor.  The host supplies Pillow's coefficient tables restricted to the crop
 * window (omnidata_b200/imageproc.py): bounds_* int32 [n][2] = (first source index, tap count),
 * kk_* int32 [n][ksize_*] fixed-point weights; bounds_h / kk_h for the out_w kept columns, bounds_v / kk_v
 * for the out_h kept rows; the horizontal pass runs over source rows [row0, row0 + nrows) into
 * tmp (uint8 [nrows][out_w][channels]).  out: fp32 [3][out_h][out_w] = (u8 / 255 [- mean) / std]
 * (a single channel is replicated, demo.py:137-138); out_u8 (optional): the cropped 8-bit image. */
int odb_pil_resize_crop_to_tensor(const void* src, int32_t src_h, int32_t src_w, int32_t channels,
                                  int64_t src_pitch, const int32_t* bounds_h, const int32_t* kk_h,
                                  int32_t ksize_h, const int32_t* bounds_v, const int32_t* kk_v, int32_t ksize_v,
                                  int32_t row0, int32_t nrows, int32_t out_h, int32_t out_w, int32_t normalize,
                                  float mean, float stdv, void* tmp, float* out, void* out_u8, void* stream);

/* F.interpolate(x, (out_h, out_w), mode='bicubic') on fp32 planes [planes][in_h][in_w] (align_corners
 * False, A = -0.75) with the clamps of demo.py:140-145 fused: flags bit 0 = clamp the input to [0,1],
 * bit 1 = clamp the result to [0,1], bit 2 = 1 - result. */
int odb_bicubic_resize_f32(const float* in, int32_t planes, int32_t in_h, int32_t in_w, int32_t out_h,
                           int32_t out_w, int32_t flags, float* out, void* stream);

/* transforms.ToPILImage() on a float CHW tensor (demo.py:150): out uint8 [h][w][c] = trunc(x * 255);
 * clamp01 != 0 applies the reference's .clamp(0, 1) first (demo.py:140). */
int odb_f32_chw_to_u8_hwc(const float* in, int32_t c, int32_t h, int32_t w, int32_t clamp01, void* out,
                          void* stream);

/* Introspection (no GPU needed). */
int odb_abi_version(void);
const char* odb_last_error(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t odb_launch_count(void);
/* Diagnostics: when set to a device buffer of grid x (return value) uint64 slots, every following
 * odb_conv_gemm launch stamps %globaltimer at its pipeline events (prologue done, dependency wait done,
 * kernel end; per tile: MMA start / first stage full / MMA commit / epilogue start / epilogue end).
 * NULL switches it off.  Used by profiles/trace_gemm.py; never set on the product path. */
int odb_debug_conv_trace(void* device_buffer);

#ifdef __cplusplus
}
#endif
#endif /* OMNIDATA_B200_H_ */
