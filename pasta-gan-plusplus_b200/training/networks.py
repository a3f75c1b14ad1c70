"""`modulated_conv2d` -- the StyleGAN2 modulated convolution of PASTA-GAN++ -- on the B200 tensor cores.

Drop-in for the reference's training/networks.py:36-94 (same signature and argument meaning).
The reference either materialises per-sample weights and runs a `groups=batch` convolution
(fused_modconv=True) or scales activations before and after a shared-weight convolution
(fused_modconv=False); both compute

    y[n,o] = d[n,o] * sum_{i,k} w[o,i,k] * s[n,i] * x[n,i] (+ noise),   d = rsqrt(sum_{i,k} (w*s)^2 + 1e-8)

On CUDA tensors this module evaluates that expression as ONE shared-weight implicit GEMM over all
samples: the style scale s is folded into the activation packing pass, the demodulation scale d and the
noise into the GEMM epilogue, and the up=2 resampling into polyphase weights.  No per-sample weight
tensor is ever written.  `fused_modconv` therefore only selects the formulation on the differentiable /
non-CUDA composition path, as in the reference.
"""
import numpy as np
import torch

from ..torch_utils import misc
from ..torch_utils.ops import bias_act
from ..torch_utils.ops import conv2d_gradfix
from ..torch_utils.ops import conv2d_resample
from ..torch_utils.ops import fma
from ..torch_utils.ops import upfirdn2d

fused_training = True       # False: the grad-enabled CUDA path composes x * s -> conv2d_resample -> fma from separate ops (round 1)


def _kernel_path_ok(x, weight, styles, noise, up, down, padding, resample_filter):
    if not conv2d_gradfix._should_use_custom_op(x):
        return False
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (x, weight, styles, noise)):
        return False
    kh, kw = weight.shape[2:]
    if down != 1 or kh != kw or x.dtype == torch.float16:      # fp16 tensors: composition over conv2d_gradfix (native f16 MMAs)
        return False
    if up == 1:
        return isinstance(padding, int) and 0 <= padding <= kh - 1
    if up == 2:
        f = resample_filter
        return kh == 3 and padding == 1 and f is not None and f.ndim == 2 and tuple(f.shape) == (4, 4)
    return False


# up = 2 layers: per-phase transposed convolution (1x the MACs) + blur / noise / activation pass instead of the one-launch
# 4x-MAC polyphase GEMM, for layers with at least this many (out channels x in channels).  Measured at batch 32 (tools/up2_bench.py, bf16x2):
# 512->512 @32 0.91 vs 1.78 ms, 512->256 @64 1.32 vs 2.52 ms, 256->128 @128 2.26 vs 2.32 ms, 128->64 @256 3.53 vs 2.35 ms (the four passes over the
# input and the (2H+1)^2 intermediate cost more than the MACs saved once the layer is HBM-bound).
UP2_PHASES = True
UP2_PHASES_MIN_IO = 512 * 256
# below UP2_PHASES_MIN_IO and at least this: the four phases as ONE 2 x 2 GEMM with 4 * O columns (16 / 9 of the algorithmic MACs, input read once) + the
# blur pass: 256->128 @128 1.94 ms (phases 2.10, polyphase 2.35); 128->64 @256 2.80 ms (polyphase 2.43: that layer keeps the polyphase form)
UP2_TAPS4_MIN_IO = 256 * 128


def modulated_conv2d_fused_act(x, weight, styles, noise=None, up=1, padding=0, resample_filter=None, demodulate=True,
                               flip_weight=True, bias=None, act='linear', alpha=None, gain=None, clamp=None,
                               out=None, out_dtype=None, accumulate=False, memory_format=None, out_packed=None):
    """Kernel path of modulated_conv2d with bias_act fused into the same launch (what SynthesisLayer / ToRGB
    compose, networks.py:1925-1935 and SURVEY Appendix E): returns
    clamp(act(modconv(x) + bias) * gain).  Inference only (no autograd).
    x may be a conv2d_gradfix.PackedAct (then the style scale is folded into per-sample weights instead of the packing
    pass) and out_packed a PackedAct view to receive the result in operand format."""
    spec = bias_act.activation_funcs[act]
    alpha = float(spec.def_alpha if alpha is None else alpha)
    gain = float(spec.def_gain if gain is None else gain)
    clamp = float(-1 if clamp is None else clamp)
    src_dtype = torch.float32 if isinstance(x, conv2d_gradfix.PackedAct) else x.dtype
    prec = conv2d_gradfix.precision_for(src_dtype)
    _, parts = conv2d_gradfix._PRODUCTS[prec]
    e4m3 = prec == 'fp8'        # e4m3 operands; the per-phase up = 2 form keeps its intermediate in bf16
    conv2d_gradfix.check_fp8_forward_only(x if isinstance(x, torch.Tensor) else None, weight, styles, bias)
    dcoef = None
    if demodulate:
        conv2d_gradfix._init()
        dcoef = conv2d_gradfix._plugin.demod_coefs(weight, styles)
    f16 = src_dtype == torch.float16
    if up == 2:
        if f16:
            raise NotImplementedError('the fused up=2 layer takes float32 / bfloat16 tensors; call modulated_conv2d for float16')
        if (UP2_PHASES and out is None and not accumulate and padding == 1 and x.shape[2] * x.shape[3] >= 128 and
                (out_packed is not None or (out_dtype in (None, torch.float32) and memory_format in (None, torch.contiguous_format) and src_dtype == torch.float32)) and
                tuple(weight.shape[2:]) == (3, 3) and weight.shape[0] % 16 == 0 and act in ('linear', 'relu', 'lrelu') and
                (x.data.shape[0] == parts if isinstance(x, conv2d_gradfix.PackedAct) else (x.dtype == torch.float32 and x.is_contiguous())) and
                resample_filter is not None and tuple(resample_filter.shape) == (4, 4) and
                weight.shape[0] * weight.shape[1] >= min(UP2_PHASES_MIN_IO, UP2_TAPS4_MIN_IO)):
            # transposed convolution at 1x its MACs (four per-phase GEMMs) + one blur / noise / bias / activation pass on the operand format;
            # a tensor input is packed once with the style scale folded in (then the phase GEMMs use the shared weights)
            xp, st = x, styles
            if not isinstance(x, conv2d_gradfix.PackedAct):
                conv2d_gradfix._init()
                ic = x.shape[1]
                xp = conv2d_gradfix.PackedAct(conv2d_gradfix._plugin.pack_activations(x, styles, -(-ic // 64) * 64, parts, e4m3=e4m3), ic)
                st = None
            return conv2d_gradfix.up2_modconv_packed(xp, weight, st, dcoef, resample_filter, flip_weight, out_packed, noise=noise, bias=bias,
                                                     act=act, alpha=alpha, gain=gain, clamp=clamp,
                                                     taps4=weight.shape[0] * weight.shape[1] < UP2_PHASES_MIN_IO)
        pw = conv2d_gradfix.packed_up2(weight, resample_filter, flip_weight, False, parts, e4m3=e4m3)
    else:
        pw = conv2d_gradfix.packed_plain(weight, flip_weight, parts, padding, padding, f16=f16, e4m3=e4m3)
    return conv2d_gradfix.igemm_conv(x, pw, scale=styles, dcoef=dcoef, noise=noise, bias=bias, act=act, alpha=alpha,
                                     gain=gain, clamp=clamp, out=out, out_dtype=out_dtype, accumulate=accumulate,
                                     memory_format=memory_format, out_packed=out_packed)


class _FusedModulatedConv2d(torch.autograd.Function):
    """Differentiable form of the kernel path for up = down = 1 (the training-mode SynthesisLayer / ToRGB of the generator phases):

        y[n,o] = d[n,o] * conv(x[n] * s[n], W)[o] + noise            (networks.py:73-82, the reference's non-fused formulation)

    forward : ONE packing pass (x * s folded in) + ONE implicit-GEMM launch with d and the noise in its epilogue
    backward: gz = pack(gy * d);  g_xs = dgrad(gz) on the tensor cores;  (g_x, g_s) = (g_xs * s, sum_hw g_xs * x) in one reduction pass;
              g_W = wgrad(gz, packed x*s kept from the forward);  g_d = sum_hw gy * (y - noise) / d;  g_noise = sum over channels of gy.
    d itself is computed by the caller with a few tiny differentiable library ops on [N, I] x [O, I], so its dependence on W and s
    is handled by autograd.  First-order only (the reference has path-length regularisation - the only double backward through G -
    commented out, loss_fullbody.py:213-232)."""

    @staticmethod
    def forward(ctx, x, weight, styles, dcoefs, noise, padding, flip_weight):
        cg = conv2d_gradfix
        cg._init()
        prec = cg.precision_for(x.dtype)
        parts = cg._PRODUCTS[prec][1]
        o, ic, kh, kw = weight.shape
        xs = cg.PackedAct(cg._plugin.pack_activations(x, styles, cg._round_up(ic, 64), parts), ic)
        pw = cg.packed_plain(weight, flip_weight, parts, padding, padding)
        y = cg.igemm_conv(xs, pw, dcoef=dcoefs, noise=noise, precision=prec, out_dtype=x.dtype)
        need_y = dcoefs is not None and ctx.needs_input_grad[3]
        ctx.save_for_backward(x, weight, styles, dcoefs, noise, y if need_y else None)
        ctx.xs = xs if ctx.needs_input_grad[1] else None
        ctx.cfg = (padding, flip_weight, prec, parts)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        cg = conv2d_gradfix
        x, weight, styles, dcoefs, noise, y = ctx.saved_tensors
        padding, flip_weight, prec, parts = ctx.cfg
        o, ic, kh, kw = weight.shape
        gy = gy.contiguous()
        g_x = g_w = g_s = g_d = g_noise = None
        gz = cg.PackedAct(cg._plugin.pack_activations(gy, dcoefs, cg._round_up(o, 64), parts), o)      # gy * d in operand format
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[2]:
            pw_t = cg.packed_plain(weight, not flip_weight, parts, kh - 1 - padding, kw - 1 - padding, transpose_io=True)
            g_xs = cg.igemm_conv(gz, pw_t, precision=prec, out_dtype=torch.float32, out_hw=tuple(x.shape[2:]))
            xf = x if x.dtype == torch.float32 else x.float()
            g_s, g_x = cg._plugin.mul_reduce_hw(g_xs, xf, scale=styles, out_scaled=ctx.needs_input_grad[0], reduce=ctx.needs_input_grad[2])
            if g_x is not None and g_x.dtype != x.dtype:
                g_x = g_x.to(x.dtype)
            if g_s is not None:
                g_s = g_s.to(styles.dtype)
        if ctx.needs_input_grad[1] and not cg.weight_gradients_disabled:
            xs = ctx.xs if ctx.xs is not None else cg.PackedAct(cg._plugin.pack_activations(x, styles, cg._round_up(ic, 64), parts), ic)
            g_w = cg.weight_gradient(gz, xs, (o, ic, kh, kw), 1, (padding, padding), False, precision=prec, out_dtype=weight.dtype)
            if not flip_weight:
                g_w = g_w.flip([2, 3])
        ctx.xs = None
        if dcoefs is not None and ctx.needs_input_grad[3]:
            gyf = gy if gy.dtype == torch.float32 else gy.float()
            yf = y if y.dtype == torch.float32 else y.float()
            r, _ = cg._plugin.mul_reduce_hw(gyf, yf, sub=noise)
            g_d = (r / dcoefs.to(torch.float32)).to(dcoefs.dtype)
        if noise is not None and ctx.needs_input_grad[4]:
            g_noise = gy.sum(dim=(0, 1)) if noise.dim() == 2 else gy.sum(dim=1, keepdim=True)
            if noise.dim() == 4 and noise.shape[0] == 1 and gy.shape[0] > 1:
                g_noise = g_noise.sum(dim=0, keepdim=True)
            g_noise = g_noise.to(noise.dtype)
        return g_x, g_w, g_s, g_d, g_noise, None, None


def _fused_training_path_ok(x, weight, styles, noise, up, down, padding):
    """CUDA float32 / bfloat16 tensors, gradients required, stride-1 modulated convolution: the fused differentiable Function"""
    if not conv2d_gradfix._should_use_custom_op(x) or not torch.is_grad_enabled():
        return False
    if not any(t is not None and t.requires_grad for t in (x, weight, styles, noise)):
        return False
    kh, kw = weight.shape[2:]
    return (up == 1 and down == 1 and kh == kw and isinstance(padding, int) and 0 <= padding <= kh - 1 and
            x.dtype in (torch.float32, torch.bfloat16) and x.shape[2] * x.shape[3] >= 1)


@misc.profiled_function
def modulated_conv2d(
    x,                          # Input tensor of shape [batch_size, in_channels, in_height, in_width].
    weight,                     # Weight tensor of shape [out_channels, in_channels, kernel_height, kernel_width].
    styles,                     # Modulation coefficients of shape [batch_size, in_channels].
    noise           = None,     # Optional noise tensor to add to the output activations.
    up              = 1,        # Integer upsampling factor.
    down            = 1,        # Integer downsampling factor.
    padding         = 0,        # Padding with respect to the upsampled image.
    resample_filter = None,     # Low-pass filter from upfirdn2d.setup_filter().
    demodulate      = True,     # Apply weight demodulation?
    flip_weight     = True,     # False = convolution, True = correlation (matches torch.nn.functional.conv2d).
    fused_modconv   = True,     # Formulation used on the composition path (see module docstring).
):
    batch_size = x.shape[0]
    out_channels, in_channels, kh, kw = weight.shape
    misc.assert_shape(weight, [out_channels, in_channels, kh, kw])
    misc.assert_shape(x, [batch_size, in_channels, None, None])
    misc.assert_shape(styles, [batch_size, in_channels])

    if conv2d_gradfix._should_use_custom_op(x):
        conv2d_gradfix.check_fp8_forward_only(x, weight, styles, noise)
    # ---- sm_100a kernel path: one implicit GEMM, modulation / demodulation / noise fused ----
    if _kernel_path_ok(x, weight, styles, noise, up, down, padding, resample_filter):
        return modulated_conv2d_fused_act(x, weight, styles, noise=noise, up=up, padding=padding,
                                          resample_filter=resample_filter, demodulate=demodulate, flip_weight=flip_weight)

    # ---- sm_100a training path (gradients required, up = 1): the same fused launch as a differentiable Function ----
    if fused_training and _fused_training_path_ok(x, weight, styles, noise, up, down, padding):
        dcoefs = None
        if demodulate:      # d[n,o] = rsqrt(sum_i s[n,i]^2 * sum_k w[o,i,k]^2 + 1e-8): tiny differentiable library ops
            w2 = weight.to(torch.float32).square().sum(dim=[2, 3])
            dcoefs = (styles.to(torch.float32).square() @ w2.t() + 1e-8).rsqrt()
        return _FusedModulatedConv2d.apply(x, weight, styles.to(torch.float32), dcoefs, noise, padding, bool(flip_weight))

    # ---- composition path (differentiable; any device): the reference's two formulations ----
    if x.dtype == torch.float16 and demodulate:     # pre-normalise to avoid fp16 overflow
        weight = weight * (1 / np.sqrt(in_channels * kh * kw) / weight.norm(float('inf'), dim=[1, 2, 3], keepdim=True))
        styles = styles / styles.norm(float('inf'), dim=1, keepdim=True)
    w = dcoefs = None
    if demodulate or fused_modconv:
        w = weight.unsqueeze(0) * styles.reshape(batch_size, 1, -1, 1, 1)           # [N, O, I, kh, kw]
    if demodulate:
        dcoefs = (w.square().sum(dim=[2, 3, 4]) + 1e-8).rsqrt()                     # [N, O]
    use_grouped = fused_modconv and not conv2d_gradfix._should_use_custom_op(x)     # grouped conv only via the library
    if not use_grouped:
        x = x * styles.to(x.dtype).reshape(batch_size, -1, 1, 1)
        x = conv2d_resample.conv2d_resample(x=x, w=weight.to(x.dtype), f=resample_filter, up=up, down=down,
                                            padding=padding, flip_weight=flip_weight)
        if demodulate and noise is not None:
            x = fma.fma(x, dcoefs.to(x.dtype).reshape(batch_size, -1, 1, 1), noise.to(x.dtype))
        elif demodulate:
            x = x * dcoefs.to(x.dtype).reshape(batch_size, -1, 1, 1)
        elif noise is not None:
            x = x.add_(noise.to(x.dtype))
        return x
    if demodulate:
        w = w * dcoefs.reshape(batch_size, -1, 1, 1, 1)
    x = x.reshape(1, -1, *x.shape[2:])
    w = w.reshape(-1, in_channels, kh, kw)
    x = conv2d_resample.conv2d_resample(x=x, w=w.to(x.dtype), f=resample_filter, up=up, down=down, padding=padding,
                                        groups=batch_size, flip_weight=flip_weight)
    x = x.reshape(batch_size, -1, *x.shape[2:])
    if noise is not None:
        x = x.add_(noise)
    return x
