/*
 * pgpp.h -- C ABI of libpgpp_sm100a.so, the prebuilt B200 (sm_100a) kernel library behind the
 * PASTA-GAN++ / StyleGAN2 synthesis ops.  It replaces the reference's ninja-JIT pybind plugins
 * (torch_utils/custom_ops.py:46-124 -> bias_act_plugin / upfirdn2d_plugin) and the cuDNN calls
 * behind conv2d_gradfix with plain `extern "C"` entry points: raw device pointers, sizes,
 * strides, scalars and a CUDA stream.  No ATen / pybind / torch types appear here.
 *
 * Conventions
 *   - every function returns 0 on success or a negative pgpp_status; pgpp_last_error() gives the
 *     message of the last failure on the calling thread (the reference raises RuntimeError through
 *     TORCH_CHECK, bias_act.cpp:35-51, upfirdn2d.cpp:19-36; the Python shim re-raises the same way)
 *   - inputs are borrowed and never written; outputs are caller-allocated
 *   - launches are asynchronous on `stream` (a cudaStream_t passed as void*), on the current device
 *   - the library keeps no global device state and is re-entrant
 */
#ifndef PGPP_H_
#define PGPP_H_

#include <stdint.h>

#if defined(__GNUC__)
#define PGPP_API __attribute__((visibility("default")))
#else
#define PGPP_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum { PGPP_F32 = 0, PGPP_F16 = 1, PGPP_BF16 = 2, PGPP_F64 = 3, PGPP_E4M3 = 4 } pgpp_dtype;   /* E4M3: fp8 operand format only */

typedef enum {
    PGPP_OK = 0,
    PGPP_ERR_INVALID = -1,      /* bad argument (the reference's TORCH_CHECK failures) */
    PGPP_ERR_UNSUPPORTED = -2,  /* valid but no kernel for it */
    PGPP_ERR_CUDA = -3          /* CUDA runtime / driver error */
} pgpp_status;

/* activation indices: same numbering as `cuda_idx` in torch_utils/ops/bias_act.py:23-33 */
typedef enum {
    PGPP_ACT_LINEAR = 1, PGPP_ACT_RELU = 2, PGPP_ACT_LRELU = 3, PGPP_ACT_TANH = 4, PGPP_ACT_SIGMOID = 5,
    PGPP_ACT_ELU = 6, PGPP_ACT_SELU = 7, PGPP_ACT_SOFTPLUS = 8, PGPP_ACT_SWISH = 9
} pgpp_act;

PGPP_API int pgpp_version(void);
PGPP_API const char* pgpp_last_error(void);
/* number of kernel launches issued through this library by the calling process (bench.py's gpu_launches) */
PGPP_API int64_t pgpp_launch_count(void);
/* The PGPP_* ablation switches (DESIGN.md section 5) are read from the environment once, when the library is loaded; this re-reads
 * them (timing tools that flip a switch between launches). */
PGPP_API void pgpp_refresh_env(void);

/* ---------------------------------------------------------------------------------------------
 * bias_act: y = clamp(act(x + b[(i / step_b) % size_b]) * gain), or its 1st / 2nd derivative.
 * Replaces the plugin function `bias_act(x, b, xref, yref, dy, grad, dim, act, alpha, gain, clamp)`
 * (torch_utils/ops/bias_act.cpp:32-90; kernel bias_act.cu:23-147).  All tensors are dense with the
 * same memory layout as x and `size_x` elements; b / xref / yref / dy may be NULL ("empty tensor"
 * in the reference, bias_act.py:39).  step_b = x.stride(dim) in elements.  clamp < 0 disables it.
 */
PGPP_API int pgpp_bias_act(const void* x, const void* b, const void* xref, const void* yref, const void* dy, void* y,
                  int64_t size_x, int64_t size_b, int64_t step_b, int dtype, int grad, int act,
                  float alpha, float gain, float clamp, void* stream);

/* ---------------------------------------------------------------------------------------------
 * upfirdn2d: zero-insert upsample, pad/crop, 2-D FIR, decimate.
 * Replaces the plugin function `upfirdn2d(x, f, upx, upy, downx, downy, padx0, padx1, pady0, pady1,
 * flip, gain)` (torch_utils/ops/upfirdn2d.cpp:16-94; kernels upfirdn2d.cu:29-200).
 * size/stride arrays are in PyTorch order [N, C, H, W], strides in elements (NCHW-contiguous and
 * channels_last both accepted).  f is float32 [fh, fw] with element strides f_stride_y / f_stride_x.
 * The caller computes out_size as upfirdn2d.cpp:32-33 does; padx1 / pady1 are implied by it.
 */
PGPP_API int pgpp_upfirdn2d(const void* x, const float* f, void* y,
                   const int64_t in_size[4], const int64_t in_stride[4],
                   const int64_t out_size[4], const int64_t out_stride[4],
                   int fw, int fh, int64_t f_stride_x, int64_t f_stride_y,
                   int upx, int upy, int downx, int downy, int padx0, int pady0,
                   int flip, float gain, int dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Convolution family (new; replaces F.conv2d / F.conv_transpose2d / cuDNN at
 * torch_utils/ops/conv2d_gradfix.py:38,43,112-114 and the per-sample weight algebra of
 * training/networks.py:62-70).
 */

/* d[n,o] = rsqrt(sum_{i,ky,kx} (w[o,i,ky,kx] * s[n,i])^2 + eps)   (training/networks.py:64-68).
 * w float32 [O, I, taps] contiguous, s float32 [N, I] contiguous, d float32 [N, O]. */
PGPP_API int pgpp_modconv_demod_coefs(const float* w, const float* s, float* d, int n, int o, int i, int taps,
                             float eps, void* stream);

/* Pack an activation tensor for the tensor-core path: NCHW-or-any-strided x (f32/f16/bf16/f64) ->
 * channels-innermost bf16 [parts][N][H][W][c_pad], optionally multiplied by scale[n,c] first
 * (the style modulation x * s of training/networks.py:74).  part p holds bf16(x - sum_{q<p} part q),
 * so parts = 1 is plain bf16 and parts = 2 / 3 carry 16 / 24 significand bits (error-compensated
 * fp32 mode).  Channels c >= C are zero-filled. */
PGPP_API int pgpp_pack_activations(const void* x, const int64_t size[4], const int64_t stride[4], int dtype,
                          const float* scale, void* out, int c_pad, int parts, void* stream);

/* Same, but writes channels [c_off, c_off + c_pad) of a wider channels-innermost buffer [parts][N][H][W][c_total]
 * (used to place the warped garment features next to a conv output so that `torch.cat` + 1x1 merge conv,
 * training/networks.py:2179-2181, needs no concatenation pass). */
PGPP_API int pgpp_pack_activations_slice(const void* x, const int64_t size[4], const int64_t stride[4], int dtype,
                          const float* scale, void* out, int c_pad, int c_total, int c_off, int parts, void* stream);

/* Same as pgpp_pack_activations_slice with ONE part of IEEE half instead of bfloat16 parts (operand_f16 of the conv descriptors). */
PGPP_API int pgpp_pack_activations_f16(const void* x, const int64_t size[4], const int64_t stride[4], int dtype,
                          const float* scale, void* out, int c_pad, int c_total, int c_off, void* stream);

/* Same with ONE part of e4m3 bytes (the fp8 inference precision, operand_e4m3 of the conv descriptor): unit scale, round to nearest
 * even, satfinite (|v| > 448 saturates to +-448).  c_total, c_off and c_pad are counted in channels = bytes. */
PGPP_API int pgpp_pack_activations_e4m3(const void* x, const int64_t size[4], const int64_t stride[4], int dtype,
                          const float* scale, void* out, int c_pad, int c_total, int c_off, void* stream);

/* Gradient of a bias_act that was fused into a convolution's epilogue, written straight into the operand format of the data- /
 * weight-gradient kernels: out = pgpp_pack_activations(dy * act'(.) * gain, zero where the clamp was active), act'(.) and the clamp
 * gate taken from the saved OUTPUT y - what BiasActCudaGrad.forward (bias_act.py:170-186, bias_act.cu:38-146 with grad = 1)
 * followed by a packing pass produce, bit for bit (the value is rounded through the tensor's dtype like the stored gradient is),
 * without the NCHW intermediate.  linear / relu / lrelu only (derivative from the output).  dy and y: same dtype (f32 / f16 / bf16),
 * same NCHW-like strides (pixel-contiguous).  csum (optional): float32 [N][C][pgpp_pack_act_gradient_tiles(H, W)] per-tile channel
 * sums of that gradient; their sum over N and tiles is the bias gradient (bias_act.py:135), deterministic.  f16: one IEEE-half part. */
PGPP_API int pgpp_pack_act_gradient(const void* dy, const void* y, const int64_t size[4], const int64_t stride[4], int dtype,
                          int act_fn, float alpha, float gain, float clamp, void* out, int c_pad, int parts, int f16,
                          float* csum, void* stream);
PGPP_API int pgpp_pack_act_gradient_tiles(int h, int w);

/* Per-sample modulated weights: out[n][p][row][c] = part p of bf16-split(master[row][c] * s[n][c]) for c < c_in,
 * zero for c_in <= c < c_pad (training/networks.py:65-66, w * styles).  master float32 [rows][c_pad], s float32 [N][c_in]. */
PGPP_API int pgpp_modulate_weights(const float* master, const float* s, void* out, int n, int64_t rows, int c_pad, int c_in,
                          int parts, void* stream);

/* e4m3 weight operand of the fp8 inference precision, shared (s == NULL, n == 1) or per sample (the style modulation w * s[n]):
 *   v[n][t][g][c]   = master[t][g][c] * s[n][c]   (c < c_in; zero beyond),   master float32 [taps][o_rows][c_pad]
 *   scale[n][g]     = max_{t, c} |v[n][t][g][c]| / 448                        (one scale per GEMM column; 0 for an all-zero column)
 *   out[n][t][g][c] = e4m3(v / scale[n][g])   round to nearest even, satfinite (0 where scale == 0)
 * out: n * taps * o_rows * c_pad bytes.  The convolution multiplies its accumulator by scale (pgpp_conv_desc.wscale). */
PGPP_API int pgpp_quantize_weights_e4m3(const float* master, const float* s, int n, int taps, int o_rows, int c_pad, int c_in,
                          void* out, float* scale, void* stream);

/* Weight operand packing, one launch (replaces the eager packing the round-1 Python shim did with library ops; there is no
 * reference counterpart: cuDNN consumes [O, I, kh, kw] directly at conv2d_gradfix.py:112-114):
 *   out[part][tap][o_off + row][c]  = split part `part` of  scale * W'[row, c, tap]      (zero for row / c beyond the tensor)
 *   master[tap][o_off + row][c]     = the same value in float32 (optional; start of the per-sample route, pgpp_modulate_weights)
 * w: [O, I, kh, kw] with element strides w_stride (any float dtype), or [I, O, kh, kw] with transpose_io != 0 (the
 * conv_transpose2d layout).  flip != 0 uses the spatially flipped kernel (true convolution; F.conv2d correlates).
 * phases == 1: taps = kh*kw, rows = O.  phases == 4: the StyleGAN2 up=2 layer (conv2d_resample.py:125-139) as ONE 3x3 stencil per
 * output phase (py, px): taps = 9, rows = 4 * phase_stride (row = phase * phase_stride + o),
 *   W'[phase][o, i, a, b] = 4 * sum_{fy,ky: py+fy-1-ky = 2(a-1)} sum_{fx,kx: px+fx-1-kx = 2(b-1)} k[fy,fx] * w_f[o, i, ky, kx]
 * with k the 4x4 FIR `fir` (device, float32, row-major; flipped unless flip_filter, upfirdn2d.py:193-196) and w_f the flipped /
 * unflipped kernel.  operand_f16 != 0 writes IEEE half instead of bfloat16 (parts must be 1): the fp16 layers of the
 * discriminator (networks.py:634,647) run native f16 MMAs.  The destination has o_rows rows per tap; rows outside
 * [o_off, o_off + rows) are left untouched (zero them once, or pack several tensors side by side: gamma | beta).  out may be NULL when
 * master is given (the fp8 route quantizes master with pgpp_quantize_weights_e4m3). */
PGPP_API int pgpp_pack_weights(const void* w, int w_dtype, const int64_t w_size[4], const int64_t w_stride[4], int transpose_io, int flip,
                      float scale, int phases, int phase_stride, const float* fir, int flip_filter,
                      void* out, float* master, int parts, int operand_f16, int o_rows, int o_off, int c_pad, void* stream);

/* Adjoint of the polyphase construction above: grad_weight[o, i, ky, kx] (float32 [O, I, 3, 3], storage order of the layer's
 * weight) from grad_polyphase float32 [4][O][I][3][3].  Used by the differentiable fused up=2 layer. */
PGPP_API int pgpp_up2_weight_adjoint(const float* grad_polyphase, const float* fir, int flip_filter, int flip, int o, int ic,
                            float* grad_weight, void* stream);

/* Plane reductions of the differentiable fused modulated convolution (networks.py:73-82 differentiated by hand), float32 NCHW:
 *   r[n,c]        = sum_hw a[n,c,hw] * (b[n,c,hw] - sub[n * sub_stride_n + hw])      (b NULL: 1; sub NULL: 0; r NULL: skipped)
 *   out_scaled[n,c,hw] = a[n,c,hw] * scale[n,c]                                      (out_scaled NULL: skipped; may alias a)
 * (a, b, sub) = (grad_y, y, noise): gradient of the demodulation coefficients (times dcoef);
 * (a, b, scale) = (grad of the modulated input, x, styles): style gradient and grad_x in one pass. */
/* r[n, c] = sum_{hw} a[n, c, hw] with float32 accumulation; a NCHW-contiguous float32 / float16 / bfloat16 (dtype: pgpp_dtype).
 * The bias gradients `dx.sum([0, 2, 3])` of bias_act.py:135,156 and conv2d_gradfix.py:130 are the sum over n of this. */
PGPP_API int pgpp_sum_hw(const void* a, int dtype, float* r, int n, int c, int64_t hw, void* stream);
PGPP_API int pgpp_mul_reduce_hw(const float* a, const float* b, const float* sub, int64_t sub_stride_n, const float* scale,
                       float* out_scaled, float* r, int n, int c, int64_t hw, void* stream);

/* Row-group im2col packing for convolutions with very few input channels (the 7x7 RGB stem, 3x3 convs on 1..6 channels):
 *     out[part][n][yy][x][(ry*kw + kx)*C + c] = split(x[n, c, yy - pad_y + ry, x + kx - pad_x] * scale[n,c])   (0 outside)
 * for yy in [0, H + pad_y), ry in [0, r), channels >= r*kw*C zero-filled up to 64.  The convolution then runs as a kh' =
 * ceil(kh / r), kw' = 1 implicit GEMM with vertical tap spacing r (pgpp_conv_desc.dil_y) and 64-channel operand rows, i.e.
 * r*kw times fewer MMAs and weight tiles than padding C to 64 per tap. */
PGPP_API int pgpp_pack_im2col(const void* x, const int64_t size[4], const int64_t stride[4], int dtype, const float* scale,
                          void* out, int kw, int r, int pad_x, int pad_y, int parts, void* stream);

/* SPADE modulation fused with the operand packing (training/networks.py:1713-1723 + the pre-activation of the consuming
 * Spade_Conv2dLayer, :1627-1630):
 *     v = (x - mean[n,c]) * rstd[n,c] * (1 + gamma) + beta;   if (pre_gain > 0) v = max(v, 0) * pre_gain;
 *     out[part][n][y][x][c] = bf16 split of v                  (channels c >= C zero-filled)
 * x float32 NCHW contiguous; gamma / beta float32 with NCHW-contiguous planes and a batch stride of gb_stride_n elements (so
 * they may be the two channel halves of one [N, 2C, H, W] tensor); mean / rstd float32 [N, C].  Replaces five element-wise
 * passes (instance-norm apply, 1 + gamma, multiply-add, bias_act, pack) with one. */
PGPP_API int pgpp_spade_modulate_pack(const float* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
                          int64_t gb_stride_n, void* out, int n, int c, int h, int w, int c_pad, int parts, float pre_gain, void* stream);

/* Epilogue + geometry of one implicit-GEMM convolution launch. */
typedef struct {
    /* packed activations [a_parts][N][H][W][c_pad] bf16 and packed weights [b_parts][taps][o_rows][c_pad] bf16 */
    const void* act;
    const void* wgt;
    int32_t a_parts, b_parts;
    int32_t n, h, w, c_pad;         /* input geometry; c_pad = channels consumed (multiple of 16) */
    int32_t act_pixel_stride;       /* elements between consecutive pixels of act (>= c_pad; 0 means c_pad): lets a conv read a
                                       channel slice of a wider channels-innermost buffer */
    int32_t wgt_per_sample;         /* 0: wgt is [b_parts][taps][o_rows][c_pad] shared by all samples;
                                       1: wgt is [N][b_parts][taps][o_rows][c_pad], sample n uses its own weights (the style
                                          modulation w * s[n] of training/networks.py:65-66 folded into the weights) */
    int32_t kh, kw;                 /* filter taps */
    int32_t pad_y, pad_x;           /* zero padding (top / left); bottom / right implied by out size */
    int32_t stride;                 /* 1 or 2 */
    int32_t dil_y;                  /* vertical tap spacing (0 or 1 = dense); > 1 only with stride 1 (row-group im2col operands) */
    int32_t conv_h, conv_w;         /* conv output grid (per phase) */
    int32_t o;                      /* logical output channels (per phase) */
    int32_t phases;                 /* 1, or 4 for the fused up=2 polyphase form: GEMM column g = phase*phase_stride + oc,
                                       phase = 2*py + px writes output pixel (2y+py, 2x+px) */
    int32_t phase_stride;           /* columns between phases: >= o, multiple of 16 when phases == 4 (= o when phases == 1) */
    int32_t o_rows;                 /* rows per tap in wgt: >= phases*phase_stride, multiple of block_n */
    int32_t block_n;                /* GEMM N tile: 16, 32, 64, 128 or 256 */
    int32_t products;               /* 1 (bf16), 3 (2-part split) or 6 (3-part split) */
    /* epilogue: v = acc * dcoef[n,oc] + noise[n?,y,x];  y = clamp(act(v + bias[oc]) * gain) */
    const float* dcoef;             /* [N, o] or NULL */
    const float* noise;             /* [out_h, out_w] (noise_stride_n = 0) or [N, out_h, out_w]; or NULL */
    int64_t noise_stride_n;
    const float* bias;              /* [o] or NULL */
    int32_t act_fn;                 /* pgpp_act */
    float alpha, gain, clamp;
    /* output tensor, logical [N, o, out_h, out_w] with element strides (any layout) */
    void* out;
    int32_t out_dtype;              /* PGPP_F32 / PGPP_BF16 / PGPP_F16; PGPP_E4M3 (e4m3 operands only): the channels-innermost e4m3
                                       operand format of the next conv, from the lean operand-format epilogue */
    int32_t out_h, out_w;
    int64_t out_stride[4];
    int32_t accumulate;             /* nonzero: out += result (used for `img = img + y`, networks.py:2190) */
    int32_t out_parts;              /* 1, or 2 / 3 with out_dtype BF16 and out_stride[1] == 1: write the bf16 expansion of the result
                                       (part p at out + p * out_part_stride), i.e. the packed activation format of the next conv */
    int64_t out_part_stride;
    /* SPADE epilogue (optional, spade_x != NULL; training/networks.py:1702-1723): the GEMM's o = 2C columns are gamma | beta of a
     * Spade_Norm_Block; the epilogue writes  pre_act((spade_x - mean) * rstd * (1 + gamma) + beta)  for the C channels of spade_x
     * (float32 [N, C, out_h, out_w] contiguous; mean / rstd float32 [N, C]; pre_act = relu * spade_pre_gain when spade_pre_gain > 0)
     * as channels-innermost bf16 parts (out_stride[1] == 1, out_parts 1..3).  Needs block_n == o, linear act, gain 1. */
    const float* spade_x;
    const float* spade_mean;
    const float* spade_rstd;
    float spade_pre_gain;
    int32_t operand_f16;            /* nonzero: act and wgt hold IEEE half (one part each, products == 1) instead of bfloat16 parts:
                                       the fp16 blocks of the discriminator (networks.py:634,647) on native f16 tensor-core MMAs */
    /* Instance-norm statistics of the OUTPUT fused into the epilogue (optional, stats_ws != NULL; the `param_free_norm` of
     * Spade_Norm_Block, networks.py:1702-1723, normalises what this convolution writes): every epilogue warp leaves, for its 32 pixels
     * and each output channel, a pivot value, the sum of the deviations from it and the sum of their squares:
     *     stats_ws float32 [3][M][o],  M = tiles * 4 warp partials, sample n owns rows [n * M / N, (n + 1) * M / N)
     * (no atomics: deterministic).  pgpp_instnorm_finalize turns them into mean / rstd.  Needs float32 NCHW output, one sample per
     * tile, conv_w and conv_h multiples of the pixel tile (16 x 8, or 8 x 16 in single-slab mode), o % 16 == 0, phases == 1, no
     * accumulate; pgpp_conv2d_igemm_plan reports M as stats_rows (0 = this launch cannot produce statistics). */
    float* stats_ws;
    /* fp8 inference precision (operand_e4m3 != 0): act and wgt hold ONE part of e4m3 bytes (products == 1), act at unit scale, the
     * weights of GEMM column g divided by wscale[g] (wgt_per_sample: wscale[n * o_rows + g]); the epilogue multiplies the accumulator
     * by wscale together with dcoef.  tcgen05.mma kind::f8f6f4, channel blocks of 32 / 64 / 128 channels (one byte each). */
    const float* wscale;
    int32_t operand_e4m3;
    int32_t reserved1;
} pgpp_conv_desc;

/* Implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05.mma, TMEM accumulators, TMA operand
 * loads), persistent over the SMs, with the epilogue above fused. */
PGPP_API int pgpp_conv2d_igemm(const pgpp_conv_desc* desc, void* stream);

/* The launch pgpp_conv2d_igemm would make for a descriptor, filled by the same validation and planning code and returned before
 * any driver call (no device needed; without one the SM count is taken as 148, the B200's). */
typedef struct {
    int32_t reuse;                  /* 0: one activation box per tap; 1: one slab per filter column (ky reuse); 2: one slab per channel block */
    int32_t slab9;                  /* single-slab mode on the straight-line 3 x 3 issuer (PGPP_IGEMM_SLAB9) */
    int32_t stack;                  /* split-precision products a0 x [b0; b1] issued as one N = 2 * block_n MMA */
    int32_t b_resident;             /* every weight tile of the column tile stays in shared memory */
    int32_t inner, n_groups;        /* taps per K group, K groups per channel block */
    int32_t parts;                  /* bf16 parts of each operand (1, 2, 3) */
    int32_t kb;                     /* channels per K block */
    int32_t tw, th, tn;             /* pixel tile: columns x rows x samples = 128 */
    int32_t block_n;
    int32_t a_stages, b_stages;     /* activation ring depth, weight slots (resident: the weight tile count) */
    int64_t total_tiles;
    int64_t grid;                   /* persistent CTAs: min(total_tiles, SM count) */
    int32_t e4m3;                   /* e4m3 operands (kind::f8f6f4) */
    int32_t epilogue;               /* 1: the lean operand-format epilogue; 0: the general one */
    int32_t fast;                   /* general epilogue on its fast path (one sample per tile, gain folded into scale / shift) */
    int32_t reserved0;
    int64_t stats_rows;             /* rows M of the instance-norm workspace (see stats_ws), 0 if the launch cannot produce statistics */
} pgpp_igemm_plan;
PGPP_API int pgpp_conv2d_igemm_plan(const pgpp_conv_desc* desc, pgpp_igemm_plan* plan);
/* mean[n, c] and rstd[n, c] = rsqrt(var + eps) (biased variance, torch.nn.InstanceNorm2d / torch.var_mean(unbiased=False)) from the
 * warp partials of pgpp_conv2d_igemm: ws float32 [3][rows][c], rows / n partials of 32 pixels per sample, merged in float64. */
PGPP_API int pgpp_instnorm_finalize(const float* ws, int64_t rows, int n, int c, float eps, float* mean, float* rstd, void* stream);

/* Masked feature composition + packing (networks.py:2253-2276, 2307-2315: the warped-garment features fed to the SPADE blocks):
 *   v[n,c,p] = x1[n,c,p]*a1[n,p] + m1[n,c]*b1[n,p]  (+ x2[n,c,p]*a2[n,p] + m2[n,c]*b2[n,p] when x2 != NULL)
 * x float32 [N,C,H,W] contiguous, m float32 [N,C], a / b float32 [N,H,W]; out = bf16 [parts][N][H][W][c_pad] (the operand format). */
PGPP_API int pgpp_mix_pack(const float* x1, const float* m1, const float* a1, const float* b1, const float* x2, const float* m2,
                  const float* a2, const float* b2, void* out, int n, int c, int h, int w, int c_pad, int parts, void* stream);

/* Direct (CUDA-core, exact float32) convolution for few-tap inputs, C * kh * kw <= 16, kw = 1 or 3, 'same' padding, stride 1 (the 3x3 conv on the
 * 1-channel parsing map of the SPADE blocks, networks.py:1702-1723; the 1x1 stem on the 5-channel pose map, :357-371):
 *   y = clamp(act(conv(x, w * wscale) + bias) * gain)
 * x float32 [N,C,H,W] contiguous, w float32 [O,C,kh,kw] contiguous; the result goes EITHER to out_nchw (float32 [N,O,H,W]) OR to
 * out_packed (bf16 operand format [parts][N][H][W][c_total], channels [c_off, c_off + O)). */
PGPP_API int pgpp_conv2d_direct(const float* x, const float* w, const float* bias, int n, int c, int h, int wd, int o, int kh, int kw,
                       int pad_y, int pad_x, float wscale, int act_fn, float alpha, float gain, float clamp,
                       float* out_nchw, void* out_packed, int c_total, int c_off, int parts, void* stream);

/* FIR blur written straight into the operand format (conv2d_resample.py:119-122, "blur, then strided convolution", without the
 * float32 intermediate): upfirdn2d with up = down = 1 and a filter of at most 4 x 4 on x (float32 [N,C,H,W], unit stride along W,
 * element strides given) -> bf16 [parts][N][H'][W'][c_pad], H' = H + pady0 + pady1 - fh + 1.  f is a HOST array of fh * fw taps. */
PGPP_API int pgpp_fir_pack(const float* x, const int64_t size[4], const int64_t stride[4], const float* f_host, int fw, int fh,
                  int padx0, int padx1, int pady0, int pady1, int flip, float gain, void* out, int c_pad, int parts, void* stream);

/* 1x1 modulated convolution with at most 8 output channels (o1 + o2) per launch on the operand format (the ToRGB layers, networks.py:1925-1967; with the
 * 7-channel parsing head of ToRGBLayerFull_v1_v5 as a second head computed in the same pass over x):
 *   out[n, o, p] (+)= clamp(act(sum_c X[n, p, c] * w[o, c] * styles[n, c] + b[o]) * gain),  X = sum of the x_parts bf16 parts.
 * x: bf16 [x_parts][N][hw][c_total] (pointer at the first of the c channels); w1 [o1, c], w2 [o2, c] float32; styles [N, c] or NULL;
 * out1 [N, o1, hw] float32 (accumulate1: added to its previous content), out2 [N, o2, hw] float32 (o2 may be 0).
 * act_fn linear / relu / lrelu.  Bound by reading x once: runs on the CUDA cores. */
PGPP_API int pgpp_conv1x1_thin(const void* x, int x_parts, int64_t x_part_stride, int c_total, int n, int c, int64_t hw,
                      const float* w1, const float* b1, int o1, float* out1, int accumulate1,
                      const float* w2, const float* b2, int o2, float* out2,
                      const float* styles, int act_fn, float alpha, float gain, float clamp, void* stream);

/* upfirdn2d with up = 1 on the operand format, packed -> packed (the blur of "blur, then strided convolution", conv2d_resample.py:119-122,
 * and the FIR decimation before a 1x1 down-sampling convolution, :107-110, for inputs whose producer already wrote the operand format):
 *   out = split_bf16( gain * sum_{jy,jx} X[n][oy*down + jy - pady0][ox*down + jx - padx0][c] * k[jy][jx] ),  X = sum of the input parts,
 * k = f flipped unless `flip` (upfirdn2d.py:193-196).  in: bf16 [in_parts][N][H][W][in_c_total] (pointer at the first of the c channels),
 * out: bf16 [out_parts][N][H'][W'][out_c_total], H' = (H + pady0 + pady1 - fh) / down + 1.  c % 8 == 0, filter at most 4 x 4 (HOST array
 * of fh * fw taps, NULL = the identity for fw * fh == 1: a channel-slice copy), down 1 or 2. */
PGPP_API int pgpp_fir_packed(const void* in, int in_parts, int64_t in_part_stride, int n, int h, int w, int c, int in_c_total,
                    const float* f_host, int fw, int fh, int down, int padx0, int padx1, int pady0, int pady1, int flip, float gain,
                    void* out, int out_parts, int64_t out_part_stride, int out_c_total, void* stream);
/* The same FIR (down = 1, separable filter) followed by  v = clamp(act(v + noise[n?, y, x] + bias[c]) * act_gain):  the blur + noise + bias_act tail of
 * the StyleGAN2 up = 2 layer (conv2d_resample.py:125-139 transposed convolution -> upfirdn2d, then networks.py:1925-1935) when the transposed
 * convolution wrote its (2H + 1) x (2W + 1) result in the operand format.  noise float32 [oh, ow] (noise_stride_n = 0) or [N, oh, ow], or NULL;
 * bias float32 [c] or NULL; act_fn linear / relu / lrelu.  The result goes EITHER to out (operand format) OR, with out == NULL, to out_nchw
 * (float32 [N, c_out, oh, ow] contiguous, c_out <= c: the low-resolution blocks hand tensors over). */
PGPP_API int pgpp_fir_packed_act(const void* in, int in_parts, int64_t in_part_stride, int n, int h, int w, int c, int in_c_total,
                    const float* f_host, int fw, int fh, int padx0, int padx1, int pady0, int pady1, int flip, float gain,
                    const float* noise, int64_t noise_stride_n, const float* bias, int act_fn, float alpha, float act_gain, float clamp,
                    void* out, int out_parts, int64_t out_part_stride, int out_c_total, float* out_nchw, int c_out, void* stream);

/* ---- weight gradient (conv2d_gradfix.py:135-142, Conv2dGradWeight.forward: replaces
 * aten::cudnn_convolution_backward_weight / cudnn_convolution_transpose_backward_weight) ----
 *
 *   G[a, b, ky, kx] = sum_{n, y, x} S[n, a, y, x] * L[n, b, y*stride + ky - pad_y, x*stride + kx - pad_x]
 *
 * conv2d:           S = grad_output, L = input        -> G = dW[O, I, kh, kw]
 * conv_transpose2d: S = input,       L = grad_output  -> G = dW[I, O, kh, kw]
 * Both operands are channels-innermost packed activations (pgpp_pack_activations: bf16 [parts][N][H][W][c_pad],
 * channels beyond C zero), the same format the forward kernel consumes. */

typedef struct pgpp_wgrad_desc {
    const void* small;              /* S: bf16 [s_parts][N][hs][ws][s_pixel_stride] */
    const void* large;              /* L: bf16 [l_parts][N][hl][wl][l_pixel_stride] */
    int32_t s_parts, l_parts;
    int32_t n;
    int32_t ca, ca_pad, s_pixel_stride;     /* channels of S, padded count (multiple of 64), elements between pixels (0: ca_pad) */
    int32_t hs, ws;
    int32_t cb, cb_pad, l_pixel_stride;
    int32_t hl, wl;
    int32_t kh, kw, pad_y, pad_x;
    int32_t stride;                 /* 1 or 2 */
    int32_t products;               /* 1 (bf16), 3 (2-part split) or 6 (3-part split) */
    float* out;                     /* G: float32 [ca][cb][kh][kw], overwritten */
    float* workspace;               /* float32 [kh*kw][ca][cb_pad] scratch (split-K partial sums land here), 16-byte aligned */
    int32_t operand_f16;            /* nonzero: S and L hold IEEE half (one part, products == 1) instead of bfloat16 parts */
    int32_t dil_y;                  /* vertical tap spacing (0 or 1 = dense): tap ky reads L row y + ky * dil_y - pad_y; > 1 with stride 1 only - the
                                       weight gradient of a convolution that ran on a row-group im2col operand (pgpp_pack_im2col) */
    float out_scale;                /* G is multiplied by this on its way out of the workspace (0 = 1): the runtime weight gain of the reference's
                                       layers, d(w * gain)/dw (networks.py:169), without a pass of its own */
    int32_t reserved0;
} pgpp_wgrad_desc;

/* Split-K GEMM over the pixels on the 5th-gen tensor cores (tcgen05.mma, TMEM accumulators, TMA operand loads). */
PGPP_API int pgpp_conv2d_wgrad(const pgpp_wgrad_desc* desc, void* stream);

/* ---- input / output edge of the try-on inference loop (test.py:126-147, :162-166) ----
 *
 * src uint8 [N, C, H*W] contiguous -> channels [c_off, c_off + C) of dst float32 [N, dst_c_total, H*W]:
 *   normalize != 0: x / 127.5 - 1 (test.py:126-140), else a plain cast (masks, test.py:139,142);
 *   mask (float32 [N, 1, H*W] or NULL): then x * mask - (1 - mask), the retain composition of test.py:144.
 * Separately rounded IEEE operations: bit-identical to the reference's torch expressions. */
PGPP_API int pgpp_u8_to_f32(const void* src, int64_t n, int64_t c, int64_t hw, void* dst, int64_t dst_c_total, int64_t c_off,
                   int normalize, const float* mask, void* stream);

/* img float32 [N, C, H*W] -> out uint8 [N, H*W, C] = trunc(clip((x + 1) * 127.5, 0, 255)), channel order reversed when
 * reverse_channels != 0 (RGB -> BGR, test.py:162-166). */
PGPP_API int pgpp_image_to_u8(const float* img, int64_t n, int64_t c, int64_t hw, void* out, int reverse_channels, void* stream);

/* ---- grid_sample (torch_utils/ops/grid_sample_gradfix.py:27-83): 2-D, bilinear, zeros padding, align_corners = False ----
 * input float32 [N,C,H,W] contiguous, grid float32 [N,Ho,Wo,2] contiguous (x, y in [-1, 1]), out float32 [N,C,Ho,Wo].
 * Replaces aten::grid_sampler_2d (grid_sample_gradfix.py:49). */
PGPP_API int pgpp_grid_sample_2d(const float* input, const float* grid, float* out, int n, int c, int h, int w, int ho, int wo, void* stream);

/* Replaces aten::grid_sampler_2d_backward (grid_sample_gradfix.py:64-65).  grad_input [N,C,H,W] (zeroed here, scatter-add) and / or
 * grad_grid [N,Ho,Wo,2]; pass NULL for the one that is not needed. */
PGPP_API int pgpp_grid_sample_2d_backward(const float* grad_out, const float* input, const float* grid, float* grad_input, float* grad_grid,
                                 int n, int c, int h, int w, int ho, int wo, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PGPP_H_ */
