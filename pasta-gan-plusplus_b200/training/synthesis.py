"""The callers of the hot path: the StyleGAN2 synthesis layers of the PASTA-GAN++ generator, written
against this package's ops.  Parameter / buffer names and shapes follow the reference so its
checkpoints map one-to-one (SURVEY.md section 5, "Checkpoint / resume"):

    FullyConnectedLayer  training/networks.py:99-128
    Conv2dLayer          training/networks.py:133-179
    SynthesisLayer       upstream StyleGAN2-ADA class the reference relies on but does not ship
                         (SURVEY.md E3 / Appendix E item 4)
    ToRGBLayer           training/networks.py:1939-1967 (ToRGBLayerFull_v1_v5, optional 7-channel parsing head)
    SynthesisBlock       training/networks.py:2086-2194 (SynthesisBlockFull_v1_v6, 'skip' architecture)
    SynthesisChain       the block sequence b8..b512 plus the texture-branch block of
                         SynthesisNetworkFull_v18 (training/networks.py:2198-2327) WITHOUT the SPADE
                         refinement blocks (out of scope this round, SURVEY.md section 8f N1)

Every layer has two routes that compute the same thing:
  fused=True   inference on CUDA: one implicit-GEMM launch per layer with modulation, demodulation,
               noise, bias, activation, gain and clamp in its prologue/epilogue (ToRGB additionally
               accumulates into the up-sampled skip image in place)
  fused=False  the drop-in composition: modulated_conv2d(...) then bias_act(...), exactly the calls the
               reference model makes (differentiable; any device with impl='ref').
"""
import numpy as np
import torch

from ..torch_utils.ops import bias_act
from ..torch_utils.ops import conv2d_gradfix
from ..torch_utils.ops import conv2d_resample
from ..torch_utils.ops import upfirdn2d
from .networks import modulated_conv2d, modulated_conv2d_fused_act


PackedAct = conv2d_gradfix.PackedAct
PACKED_MIN_RES = 128    # blocks at this resolution and above hand activations over in operand format (no packing passes)


# pgpp_fir_pack (one pass: blur -> operand format) measured 2.57 ms for 32x64x512x512 against 1.18 + 0.75 ms for the blur kernel
# followed by the packing kernel (profiles/r01_pack_bench_v15.txt): its 64-channel x 128-pixel tile pays a 1.9x halo and a long
# staging loop.  Kept for comparison, off by default.
FUSE_BLUR_PACK = False
THIN_TORGB = True       # ToRGB (and its parsing head) on operand-format inputs: one pass of the bandwidth-bound pgpp_conv1x1_thin kernel


def _can_fuse(x, *params):
    if isinstance(x, PackedAct):
        return True
    if not conv2d_gradfix._should_use_custom_op(x):
        return False
    return not (torch.is_grad_enabled() and any(p is not None and p.requires_grad for p in (x,) + params))


def _parts():
    # 'fp8': the hand-over format stays one bf16 part; every implicit GEMM converts its operand to e4m3 (conv2d_gradfix.e4m3_operand)
    return conv2d_gradfix._PRODUCTS[conv2d_gradfix.fp32_precision][1]


def _register(module, name, value, trainable):
    """frozen layers keep their tensors as BUFFERS (networks.py:153-162): same state-dict names, but absent from `parameters()`, so
    neither `module.requires_grad_(True)` at the start of a phase nor the optimiser or DDP ever touches them"""
    if value is None:
        setattr(module, name, None)
    elif trainable:
        setattr(module, name, torch.nn.Parameter(value))
    else:
        module.register_buffer(name, value)


class FullyConnectedLayer(torch.nn.Module):
    def __init__(self, in_features, out_features, bias=True, activation='linear', lr_multiplier=1, bias_init=0, trainable=True):
        super().__init__()
        self.activation = activation
        _register(self, 'weight', torch.randn([out_features, in_features]) / lr_multiplier, trainable)
        _register(self, 'bias', torch.full([out_features], np.float32(bias_init)) if bias else None, trainable)
        self.weight_gain = lr_multiplier / np.sqrt(in_features)
        self.bias_gain = lr_multiplier

    def forward(self, x, impl='cuda'):
        w = self.weight.to(x.dtype) * self.weight_gain
        b = self.bias
        if b is not None:
            b = b.to(x.dtype)
            if self.bias_gain != 1:
                b = b * self.bias_gain
        if self.activation == 'linear' and b is not None:
            return torch.addmm(b.unsqueeze(0), x, w.t())        # plain library GEMM (cuBLAS), as in the reference
        return bias_act.bias_act(x.matmul(w.t()), b, act=self.activation, impl=impl)


class Conv2dLayer(torch.nn.Module):
    def __init__(self, in_channels, out_channels, kernel_size, bias=True, activation='linear', up=1, down=1,
                 resample_filter=[1, 3, 3, 1], conv_clamp=None, channels_last=False, trainable=True):
        super().__init__()
        self.activation = activation
        self.up, self.down = up, down
        self.conv_clamp = conv_clamp
        self.register_buffer('resample_filter', upfirdn2d.setup_filter(resample_filter))
        self.padding = kernel_size // 2
        self.weight_gain = 1 / np.sqrt(in_channels * (kernel_size ** 2))
        self.act_gain = bias_act.activation_funcs[activation].def_gain
        _register(self, 'weight', torch.randn([out_channels, in_channels, kernel_size, kernel_size]), trainable)
        _register(self, 'bias', torch.zeros([out_channels]) if bias else None, trainable)

    def forward(self, x, gain=1, fused=True, impl='cuda', out_packed=None, out=None, accumulate=False):
        """`out_packed=`: write the operand format of the next convolution instead of an NCHW tensor; `out=` / `accumulate=`: write
        (or add, `y = skip + conv1(...)` of the residual blocks) into an existing NCHW float32 tensor.  Fused route only."""
        act_gain = self.act_gain * gain
        act_clamp = self.conv_clamp * gain if self.conv_clamp is not None else None
        if fused and self.up == 1 and self.down == 1 and _can_fuse(x, self.weight, self.bias) and not isinstance(x, PackedAct) and \
                x.dtype == torch.float32 and out is None and self.padding * 2 == self.weight.shape[-1] - 1 and \
                conv2d_gradfix.direct_conv_ok(self.weight, self.activation):
            # few-tap stem (e.g. 1x1 on the 5-channel pose map): exact-fp32 direct kernel, bound by writing its output
            return conv2d_gradfix.direct_conv(x, self.weight, self.bias, wscale=self.weight_gain, act=self.activation,
                                              alpha=bias_act.activation_funcs[self.activation].def_alpha, gain=act_gain,
                                              clamp=-1 if act_clamp is None else act_clamp, out_packed=out_packed)
        if fused and self.up == 1 and self.down == 1 and _can_fuse(x, self.weight, self.bias):
            parts = _parts() if isinstance(x, PackedAct) else conv2d_gradfix._PRODUCTS[conv2d_gradfix.precision_for(x.dtype)][1]
            f16 = (not isinstance(x, PackedAct)) and x.dtype == torch.float16                     # fp16 blocks of the discriminator
            im2col = (not isinstance(x, PackedAct)) and x.shape[2] >= 8 and x.shape[3] >= 16 and not f16      # few-channel stems (7x7 RGB, 3x3 on 6 ch)
            pw = conv2d_gradfix.packed_plain(self.weight, True, parts, self.padding, self.padding, scale=self.weight_gain, allow_im2col=im2col,
                                             f16=f16)
            return conv2d_gradfix.igemm_conv(x, pw, bias=self.bias, act=self.activation,
                                             alpha=bias_act.activation_funcs[self.activation].def_alpha, gain=act_gain,
                                             clamp=-1 if act_clamp is None else act_clamp, out_packed=out_packed, out=out,
                                             accumulate=accumulate)
        assert out is None and not accumulate, 'out= / accumulate= need the fused stride-1 route'
        if fused and self.up == 1 and self.down == 2 and isinstance(x, PackedAct):
            # operand-format input: the FIR runs on that format too (pgpp_fir_packed), no float32 intermediate and no packing pass
            k = self.weight.shape[-1]
            fw = self.resample_filter.shape[-1]
            p0 = self.padding + (fw - 2 + 1) // 2
            p1 = self.padding + (fw - 2) // 2
            pw = conv2d_gradfix.packed_plain(self.weight, True, _parts(), 0, 0, scale=self.weight_gain)
            epi = dict(bias=self.bias, act=self.activation, alpha=bias_act.activation_funcs[self.activation].def_alpha, gain=act_gain,
                       clamp=-1 if act_clamp is None else act_clamp)
            if k == 1:
                xd = conv2d_gradfix.fir_packed(x, self.resample_filter, down=2, padding=(p0, p1, p0, p1))
                return conv2d_gradfix.igemm_conv(xd, pw, out_packed=out_packed, **epi)
            xb = conv2d_gradfix.fir_packed(x, self.resample_filter, down=1, padding=(p0, p1, p0, p1))
            return conv2d_gradfix.igemm_conv(xb, pw, stride=2, out_packed=out_packed, **epi)
        if fused and self.up == 1 and self.down == 2 and _can_fuse(x, self.weight, self.bias) and not isinstance(x, PackedAct):
            # FIR blur (or FIR decimation for 1x1 kernels) on the upfirdn2d kernel, then ONE strided implicit-GEMM launch with the
            # bias / activation fused (conv2d_resample.py:107-110, 119-122)
            k = self.weight.shape[-1]
            fw = self.resample_filter.shape[-1]
            p0 = self.padding + (fw - 2 + 1) // 2
            p1 = self.padding + (fw - 2) // 2
            parts = conv2d_gradfix._PRODUCTS[conv2d_gradfix.precision_for(x.dtype)][1]
            pw = conv2d_gradfix.packed_plain(self.weight, True, parts, 0, 0, scale=self.weight_gain, f16=x.dtype == torch.float16)
            epi = dict(bias=self.bias, act=self.activation, alpha=bias_act.activation_funcs[self.activation].def_alpha, gain=act_gain,
                       clamp=-1 if act_clamp is None else act_clamp)
            if k == 1:
                x = upfirdn2d.upfirdn2d(x, self.resample_filter, down=2, padding=[p0, p1, p0, p1])
                return conv2d_gradfix.igemm_conv(x, pw, out_packed=out_packed, **epi)
            if FUSE_BLUR_PACK and x.dtype == torch.float32 and x.stride(3) == 1 and self.resample_filter.ndim == 2 and fw <= 4:
                # blur written straight into the operand format of the strided GEMM (no float32 intermediate, no packing pass)
                if getattr(self, '_filter_host', None) is None:
                    self._filter_host = [float(v) for v in self.resample_filter.detach().cpu().reshape(-1)]     # one sync, first call only
                conv2d_gradfix._init()
                ic = x.shape[1]
                data = conv2d_gradfix._plugin.fir_pack(x, self._filter_host, fw, fw, p0, p1, p0, p1, False, 1.0, pw.c_pad, parts)
                return conv2d_gradfix.igemm_conv(PackedAct(data, ic), pw, stride=2, out_packed=out_packed, **epi)
            # blurred image of odd width (2W' + 1): rows padded to 16 bytes so the FIR stores and the packing loads stay 128-bit
            upfirdn2d._init()
            x = upfirdn2d._plugin.upfirdn2d(x, self.resample_filter, 1, 1, 1, 1, p0, p1, p0, p1, False, 1.0, row_align=4)
            return conv2d_gradfix.igemm_conv(x, pw, stride=2, out_packed=out_packed, **epi)
        assert out_packed is None and not isinstance(x, PackedAct)
        b = self.bias.to(x.dtype) if self.bias is not None else None
        if conv2d_gradfix._should_use_custom_op(x) and self.weight.dtype == torch.float32:
            # kernel path (training): the runtime gain and the cast are folded into the packed copy of the PARAMETER, which is then made
            # once per optimizer step instead of once per call from the temporary `weight * gain` (networks.py:169)
            if impl == 'cuda':      # bias / activation / gain / clamp in the convolution's epilogue where the decomposition allows
                return conv2d_resample.conv2d_resample(x=x, w=self.weight, f=self.resample_filter, up=self.up, down=self.down,
                                                       padding=self.padding, flip_weight=(self.up == 1), w_scale=float(self.weight_gain),
                                                       bias_act_args=dict(b=b, act=self.activation, gain=act_gain, clamp=act_clamp))
            x = conv2d_resample.conv2d_resample(x=x, w=self.weight, f=self.resample_filter, up=self.up, down=self.down,
                                                padding=self.padding, flip_weight=(self.up == 1), w_scale=float(self.weight_gain))
        else:
            w = self.weight * self.weight_gain
            x = conv2d_resample.conv2d_resample(x=x, w=w.to(x.dtype), f=self.resample_filter, up=self.up, down=self.down,
                                                padding=self.padding, flip_weight=(self.up == 1))
        return bias_act.bias_act(x, b, act=self.activation, gain=act_gain, clamp=act_clamp, impl=impl)


class SynthesisLayer(torch.nn.Module):
    def __init__(self, in_channels, out_channels, w_dim, resolution, kernel_size=3, up=1, use_noise=True,
                 activation='lrelu', resample_filter=[1, 3, 3, 1], conv_clamp=None):
        super().__init__()
        self.resolution = resolution
        self.up = up
        self.use_noise = use_noise
        self.activation = activation
        self.conv_clamp = conv_clamp
        self.register_buffer('resample_filter', upfirdn2d.setup_filter(resample_filter))
        self.padding = kernel_size // 2
        self.act_gain = bias_act.activation_funcs[activation].def_gain
        self.affine = FullyConnectedLayer(w_dim, in_channels, bias_init=1)
        self.weight = torch.nn.Parameter(torch.randn([out_channels, in_channels, kernel_size, kernel_size]))
        if use_noise:
            self.register_buffer('noise_const', torch.randn([resolution, resolution]))
            self.noise_strength = torch.nn.Parameter(torch.zeros([]))
        self.bias = torch.nn.Parameter(torch.zeros([out_channels]))

    def forward(self, x, w, noise_mode='random', fused_modconv=True, gain=1, fused=True, impl='cuda', out_packed=None):
        assert noise_mode in ['random', 'const', 'none']
        styles = self.affine(w)
        noise = None
        if self.use_noise and noise_mode == 'random':
            noise = torch.randn([x.shape[0], 1, self.resolution, self.resolution], device=x.device) * self.noise_strength
        if self.use_noise and noise_mode == 'const':
            noise = self.noise_const * self.noise_strength
        flip_weight = (self.up == 1)
        act_gain = self.act_gain * gain
        act_clamp = self.conv_clamp * gain if self.conv_clamp is not None else None
        if fused and _can_fuse(x, self.weight, self.bias, styles, noise):
            return modulated_conv2d_fused_act(x, self.weight, styles, noise=noise, up=self.up, padding=self.padding,
                                              resample_filter=self.resample_filter, flip_weight=flip_weight, bias=self.bias,
                                              act=self.activation, gain=act_gain, clamp=act_clamp, out_packed=out_packed)
        assert out_packed is None and not isinstance(x, PackedAct)
        x = modulated_conv2d(x=x, weight=self.weight, styles=styles, noise=noise, up=self.up, padding=self.padding,
                             resample_filter=self.resample_filter, flip_weight=flip_weight, fused_modconv=fused_modconv)
        return bias_act.bias_act(x, self.bias.to(x.dtype), act=self.activation, gain=act_gain, clamp=act_clamp, impl=impl)


class ToRGBLayer(torch.nn.Module):
    def __init__(self, in_channels, out_channels, w_dim, kernel_size=1, conv_clamp=None, parsing_channels=0):
        super().__init__()
        self.conv_clamp = conv_clamp
        self.affine = FullyConnectedLayer(w_dim, in_channels, bias_init=1)
        self.weight = torch.nn.Parameter(torch.randn([out_channels, in_channels, kernel_size, kernel_size]))
        self.bias = torch.nn.Parameter(torch.zeros([out_channels]))
        self.weight_gain = 1 / np.sqrt(in_channels * (kernel_size ** 2))
        if parsing_channels:
            self.m_weight1 = torch.nn.Parameter(torch.randn([parsing_channels, in_channels, kernel_size, kernel_size]))
            self.m_bias1 = torch.nn.Parameter(torch.zeros([parsing_channels]))
        self.parsing_channels = parsing_channels

    def forward(self, x, w, fused_modconv=True, img=None, fused=True, impl='cuda'):
        """Returns (rgb, pred_parsing); when `img` is given the fused route adds rgb into it in place
        (`img.add_(y)`, networks.py:2190) and returns img."""
        styles = self.affine(w) * self.weight_gain
        pred_parsing = None
        can = fused and _can_fuse(x, self.weight, self.bias, styles)
        if can and THIN_TORGB and isinstance(x, PackedAct) and tuple(self.weight.shape[2:]) == (1, 1) and x.c % 8 == 0 and x.c <= 512 and \
                self.weight.shape[0] + self.parsing_channels <= 16 and (img is None or (img.dtype == torch.float32 and img.is_contiguous())):
            # operand-format input: both heads (RGB and parsing) from ONE pass over x on the bandwidth-bound thin kernel
            conv2d_gradfix._init()
            n, ic, h, wd = x.shape
            oc = self.weight.shape[0]
            y = img if img is not None else torch.empty([n, oc, h, wd], dtype=torch.float32, device=x.device)
            clamp = -1.0 if self.conv_clamp is None else float(self.conv_clamp)
            w2 = b2 = None
            if self.parsing_channels:
                pred_parsing = torch.empty([n, self.parsing_channels, h, wd], dtype=torch.float32, device=x.device)
                w2, b2 = self.m_weight1.reshape(self.parsing_channels, ic), self.m_bias1
                if oc + self.parsing_channels > 8:      # one launch holds 8 outputs' weights in registers: the parsing head takes its own pass
                    conv2d_gradfix._plugin.conv1x1_thin(x.data, ic, x.c_off, w2, b2, pred_parsing, False, styles=styles, clamp=clamp)
                    w2 = b2 = None
            conv2d_gradfix._plugin.conv1x1_thin(x.data, ic, x.c_off, self.weight.reshape(oc, ic), self.bias, y, img is not None, w2=w2, b2=b2,
                                                out2=pred_parsing if w2 is not None else None, styles=styles, clamp=clamp)
            return y, pred_parsing
        if self.parsing_channels:
            if can:
                pred_parsing = modulated_conv2d_fused_act(x, self.m_weight1, styles, demodulate=False, bias=self.m_bias1,
                                                          clamp=self.conv_clamp)
            else:
                pred_parsing = modulated_conv2d(x=x, weight=self.m_weight1, styles=styles, demodulate=False, fused_modconv=fused_modconv)
                pred_parsing = bias_act.bias_act(pred_parsing, self.m_bias1.to(x.dtype), clamp=self.conv_clamp, impl=impl)
        if can:
            y = modulated_conv2d_fused_act(x, self.weight, styles, demodulate=False, bias=self.bias, clamp=self.conv_clamp,
                                           out=img, accumulate=img is not None, out_dtype=torch.float32,
                                           memory_format=torch.contiguous_format)
            return y, pred_parsing
        assert not isinstance(x, PackedAct)
        y = modulated_conv2d(x=x, weight=self.weight, styles=styles, demodulate=False, fused_modconv=fused_modconv)
        y = bias_act.bias_act(y, self.bias.to(x.dtype), clamp=self.conv_clamp, impl=impl)
        y = y.to(dtype=torch.float32, memory_format=torch.contiguous_format)
        if img is not None:
            y = img.add_(y)
        return y, pred_parsing


class SynthesisBlock(torch.nn.Module):
    def __init__(self, in_channels, out_channels, w_dim, resolution, img_channels, is_last=False, parsing_channels=0,
                 resample_filter=[1, 3, 3, 1], conv_clamp=None, merge_channels=64, use_noise=True):
        super().__init__()
        self.in_channels = in_channels
        self.resolution = resolution
        self.img_channels = img_channels
        self.register_buffer('resample_filter', upfirdn2d.setup_filter(resample_filter))
        self.num_conv = 0
        self.num_torgb = 1
        if in_channels != 0:
            self.conv0 = SynthesisLayer(in_channels, out_channels, w_dim=w_dim, resolution=resolution, up=2,
                                        resample_filter=resample_filter, conv_clamp=conv_clamp, use_noise=use_noise)
            self.num_conv += 1
        self.conv1 = SynthesisLayer(out_channels, out_channels, w_dim=w_dim, resolution=resolution, conv_clamp=conv_clamp,
                                    use_noise=use_noise)
        self.num_conv += 1
        self.torgb = ToRGBLayer(out_channels, img_channels, w_dim=w_dim, conv_clamp=conv_clamp,
                                parsing_channels=parsing_channels if is_last else 0)
        if resolution > 32 and merge_channels:
            self.merge_conv = Conv2dLayer(out_channels + merge_channels, out_channels, kernel_size=1, resample_filter=resample_filter)

    def forward(self, x, img, ws, pose_feature=None, cat_feat=None, fused=True, impl='cuda', **layer_kwargs):
        """x: previous block's feature map as a tensor or (from blocks >= PACKED_MIN_RES on the fused route) a PackedAct.
        Returns (x, img, pred_parsing); x is a PackedAct when this block ran in operand-format hand-over mode."""
        w_iter = iter(ws.unbind(dim=1))
        merge = hasattr(self, 'merge_conv') and cat_feat is not None
        if self.in_channels == 0:
            x = self.conv1(pose_feature.to(torch.float32), next(w_iter), fused=fused, impl=impl, **layer_kwargs)
        elif fused and self.resolution >= PACKED_MIN_RES and _can_fuse(x, self.conv0.weight, self.conv1.weight) and \
                self.conv1.weight.shape[0] % 16 == 0:
            # operand-format hand-over: conv epilogues write bf16 (split) channels-innermost buffers that the next conv's
            # TMA reads directly; the garment features are packed next to conv1's output so the concat disappears
            n, res, oc, parts = ws.shape[0], self.resolution, self.conv1.weight.shape[0], _parts()
            dev = ws.device
            xa = PackedAct(PackedAct.empty(n, res, res, oc, parts, dev), oc)
            self.conv0(x, next(w_iter), fused=True, out_packed=xa, **layer_kwargs)
            if merge:
                cf = cat_feat[str(res)]
                mc = cf.shape[1]
                buf = PackedAct.empty(n, res, res, oc + mc, parts, dev)
                conv2d_gradfix._init()
                conv2d_gradfix._plugin.pack_activations_into(cf, None, buf, mc, oc)
                self.conv1(xa, next(w_iter), fused=True, out_packed=PackedAct(buf, oc, 0), **layer_kwargs)
                x = PackedAct(PackedAct.empty(n, res, res, oc, parts, dev), oc)
                self.merge_conv(PackedAct(buf, oc + mc, 0), fused=True, out_packed=x)
            else:
                x = PackedAct(PackedAct.empty(n, res, res, oc, parts, dev), oc)
                self.conv1(xa, next(w_iter), fused=True, out_packed=x, **layer_kwargs)
        else:
            x = self.conv0(x, next(w_iter), fused=fused, impl=impl, **layer_kwargs)
            x = self.conv1(x, next(w_iter), fused=fused, impl=impl, **layer_kwargs)
            if merge:
                x = torch.cat([x, cat_feat[str(x.shape[2])].to(x.dtype)], dim=1)
                x = self.merge_conv(x, fused=fused, impl=impl)
        if img is not None:
            img = upfirdn2d.upsample2d(img, self.resample_filter, impl=impl)
        img, pred_parsing = self.torgb(x, next(w_iter), img=img, fused=fused, impl=impl)
        return x, img, pred_parsing


class SynthesisChain(torch.nn.Module):
    """b8 .. b<img_resolution> main branch + the texture-branch block fed by the penultimate feature map."""

    def __init__(self, w_dim=512, img_resolution=512, img_channels=3, channel_base=32768, channel_max=512, conv_clamp=256,
                 parsing_channels=7, use_noise=True, merge_channels=64):
        super().__init__()
        assert img_resolution >= 8 and img_resolution & (img_resolution - 1) == 0
        self.w_dim = w_dim
        self.img_resolution = img_resolution
        self.block_resolutions = [2 ** i for i in range(3, int(np.log2(img_resolution)) + 1)]
        ch = {res: min(channel_base // res, channel_max) for res in self.block_resolutions}
        self.channels = ch
        self.num_ws = 0
        for res in self.block_resolutions:
            in_ch = ch[res // 2] if res > 8 else 0
            block = SynthesisBlock(in_ch, ch[res], w_dim=w_dim, resolution=res, img_channels=img_channels,
                                   is_last=(res == img_resolution), parsing_channels=parsing_channels, conv_clamp=conv_clamp,
                                   use_noise=use_noise, merge_channels=merge_channels)
            self.num_ws += block.num_conv + block.num_torgb
            setattr(self, f'b{res}', block)
        res = img_resolution
        self.texture = SynthesisBlock(ch[res // 2], ch[res], w_dim=w_dim, resolution=res, img_channels=img_channels,
                                      conv_clamp=conv_clamp, use_noise=use_noise, merge_channels=merge_channels)
        self.num_ws += self.texture.num_conv + self.texture.num_torgb

    def forward(self, ws, pose_feature, cat_feats=None, fused=True, impl='cuda', **layer_kwargs):
        """ws [N, num_ws, w_dim]; pose_feature [N, C8, 8, 8]; cat_feats {'64': [N,64,64,64], ...} or None.
        Returns (img, pred_parsing, texture_img)."""
        x = img = pred_parsing = None
        w_idx = 0
        x_prev = None
        for res in self.block_resolutions:
            block = getattr(self, f'b{res}')
            n = block.num_conv + block.num_torgb
            x_prev = x
            x, img, pp = block(x, img, ws.narrow(1, w_idx, n), pose_feature=pose_feature, cat_feat=cat_feats, fused=fused,
                               impl=impl, **layer_kwargs)
            pred_parsing = pp if pp is not None else pred_parsing
            w_idx += n
        n = self.texture.num_conv + self.texture.num_torgb
        _, tex, _ = self.texture(x_prev, None, ws.narrow(1, w_idx, n), cat_feat=cat_feats, fused=fused, impl=impl, **layer_kwargs)
        return img, pred_parsing, tex


def shard_range(total, rank, world_size):
    """Contiguous batch shard of rank `rank`: samples are independent in eval mode (SURVEY 8e), so inference shards
    by batch with no data-path collective.  Remainders go to the lowest ranks."""
    base, rem = divmod(int(total), int(world_size))
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def run_sharded(net, ws, pose_feature, cat_feats=None, rank=0, world_size=1, **kwargs):
    """Run this rank's shard of a global batch; returns ((start, stop), outputs)."""
    a, b = shard_range(ws.shape[0], rank, world_size)
    cf = None if cat_feats is None else {k: v[a:b] for k, v in cat_feats.items()}
    return (a, b), net(ws[a:b], pose_feature[a:b], cf, **kwargs)
