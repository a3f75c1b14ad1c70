"""2-D convolution with optional FIR up/down-sampling.  Drop-in for the reference's
torch_utils/ops/conv2d_resample.py (`conv2d_resample`, `_conv2d_wrapper`, same argument meaning and the
same decomposition into fast paths, conv2d_resample.py:94-154).

B200 addition: on CUDA tensors, the StyleGAN2 up=2 layer (3x3 kernel, 4x4 FIR, groups=1) runs as ONE
polyphase implicit-GEMM launch when no gradient is required -- the transposed convolution, its
(2H+1)^2 intermediate and the blur pass are folded into the weights (conv2d_gradfix.packed_up2).
"""
import torch

from .. import misc
from . import conv2d_gradfix
from . import upfirdn2d
from .upfirdn2d import _parse_padding
from .upfirdn2d import _get_filter_size


def _get_weight_shape(w):
    shape = [int(sz) for sz in w.shape]
    misc.assert_shape(w, shape)
    return shape


def _conv2d_wrapper(x, w, stride=1, padding=0, groups=1, transpose=False, flip_weight=True, w_scale=1.0, bias=None, epilogue=None):
    """conv2d / conv_transpose2d through conv2d_gradfix; flip_weight=False means true convolution."""
    _get_weight_shape(w)
    if not flip_weight:
        w = w.flip([2, 3])
    op = conv2d_gradfix.conv_transpose2d if transpose else conv2d_gradfix.conv2d
    if epilogue is not None:
        assert not transpose
        return op(x, w, bias, stride=stride, padding=padding, groups=groups, weight_scale=w_scale, epilogue=epilogue)
    if w_scale == 1.0:
        return op(x, w, stride=stride, padding=padding, groups=groups)
    return op(x, w, stride=stride, padding=padding, groups=groups, weight_scale=w_scale)


def _needs_grad(*tensors):
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


class _Pad:
    """(x0, x1, y0, y1) padding of the up-sampled image, with the bookkeeping the FIR stages add (conv2d_resample.py:96-106)"""

    def __init__(self, padding):
        self.x0, self.x1, self.y0, self.y1 = _parse_padding(padding)

    def widen(self, fw, fh, up, down):
        for factor, lo, hi in ((up, lambda t: (t + up - 1) // 2, lambda t: (t - up) // 2),
                               (down, lambda t: (t - down + 1) // 2, lambda t: (t - down) // 2)):
            if factor > 1:
                self.x0 += lo(fw); self.x1 += hi(fw)
                self.y0 += lo(fh); self.y1 += hi(fh)
        return self

    def shift(self, dx0, dx1, dy0, dy1):
        self.x0 += dx0; self.x1 += dx1; self.y0 += dy0; self.y1 += dy1
        return self

    @property
    def fir(self):              # upfirdn2d order
        return [self.x0, self.x1, self.y0, self.y1]

    @property
    def conv(self):             # F.conv2d order, valid only when symmetric
        return [self.y0, self.x0]

    @property
    def symmetric(self):
        return self.x0 == self.x1 and self.y0 == self.y1 and min(self.x0, self.y0) >= 0


def _transposed_weight(w, groups):
    """[O, I/g, kh, kw] -> the [I, O/g, kh, kw] layout conv_transpose2d expects"""
    o, ig, kh, kw = _get_weight_shape(w)
    if groups == 1:
        return w.transpose(0, 1)
    return w.reshape(groups, o // groups, ig, kh, kw).transpose(1, 2).reshape(groups * ig, o // groups, kh, kw)


@misc.profiled_function
def conv2d_resample(x, w, f=None, up=1, down=1, padding=0, groups=1, flip_weight=True, flip_filter=False, w_scale=1.0, bias_act_args=None):
    """x [N, I, H, W], w [O, I/groups, kh, kw], f from upfirdn2d.setup_filter() or None.  Padding is given
    with respect to the upsampled image and applied once.
    `w_scale` (extension): the convolution uses w * w_scale; with it `w` may be the float32 parameter itself also for a float16 x
    (see conv2d_gradfix.conv2d: the constant and the cast are folded into the cached packed copy of the parameter).
    `bias_act_args` (extension): dict(b, act, gain, clamp) of the `bias_act.bias_act` call the reference's layers make on the result
    (networks.py:172-176); the result is then that call's.  Where the decomposition ends in a convolution on the kernel path and the
    activation's gradient needs its output only, the bias / activation / gain / clamp run in that convolution's epilogue."""
    if bias_act_args is not None:
        from . import bias_act
        ba = dict(bias_act_args)
        spec = bias_act.activation_funcs[ba.get('act', 'linear')]
        # up == 1: every branch of the decomposition ends in the convolution
        if (FUSE_BIAS_ACT and up == 1 and groups == 1 and ba.get('act', 'linear') in conv2d_gradfix.FUSED_EPILOGUE_ACTS
                and conv2d_gradfix._should_use_custom_op(x)):
            epilogue = (ba.get('act', 'linear'), spec.def_alpha, spec.def_gain if ba.get('gain') is None else ba['gain'],
                        -1 if ba.get('clamp') is None else ba['clamp'])
            return _conv2d_resample(x, w, f, up, down, padding, groups, flip_weight, flip_filter, w_scale, ba.get('b'), epilogue)
        y = _conv2d_resample(x, w, f, up, down, padding, groups, flip_weight, flip_filter, w_scale, None, None)
        return bias_act.bias_act(y, ba.get('b'), act=ba.get('act', 'linear'), gain=ba.get('gain'), clamp=ba.get('clamp'))
    return _conv2d_resample(x, w, f, up, down, padding, groups, flip_weight, flip_filter, w_scale, None, None)


FUSE_BIAS_ACT = True        # False: bias_act as its own pass after the convolution (the reference's form), for comparison / tests


def _conv2d_resample(x, w, f, up, down, padding, groups, flip_weight, flip_filter, w_scale, bias, epilogue):
    assert isinstance(x, torch.Tensor) and (x.ndim == 4)
    assert isinstance(w, torch.Tensor) and (w.ndim == 4) and (w.dtype == x.dtype or (w_scale != 1.0 and w.dtype == torch.float32))
    assert f is None or (isinstance(f, torch.Tensor) and f.ndim in [1, 2] and f.dtype == torch.float32)
    assert isinstance(up, int) and (up >= 1)
    assert isinstance(down, int) and (down >= 1)
    assert isinstance(groups, int) and (groups >= 1)
    _, _, kh, kw = _get_weight_shape(w)
    fw, fh = _get_filter_size(f)
    pad = _Pad(padding)

    # fused polyphase form of the up=2 layer (inference): one implicit-GEMM launch
    if (up == 2 and down == 1 and groups == 1 and (kh, kw) == (3, 3) and f is not None and f.ndim == 2 and (fw, fh) == (4, 4)
            and pad.fir == [1, 1, 1, 1] and conv2d_gradfix._should_use_custom_op(x) and not _needs_grad(x, w) and x.dtype != torch.float16):
        prec = conv2d_gradfix.precision_for(x.dtype)
        _, parts = conv2d_gradfix._PRODUCTS[prec]
        if w_scale != 1.0:
            w = w * w_scale
        return conv2d_gradfix.igemm_conv(x, conv2d_gradfix.packed_up2(w, f, flip_weight, flip_filter, parts, e4m3=prec == 'fp8'))

    pad.widen(fw, fh, up, down)
    fir = lambda t, **kw_: upfirdn2d.upfirdn2d(x=t, f=f, flip_filter=flip_filter, **kw_)
    conv = lambda t, **kw_: _conv2d_wrapper(x=t, w=w, groups=groups, flip_weight=flip_weight, w_scale=w_scale, bias=bias, epilogue=epilogue, **kw_)
    pointwise = kh == 1 and kw == 1

    if up == 1 and down > 1:
        if pointwise:                       # decimate first, convolve the smaller image (conv2d_resample.py:107-110)
            return conv(fir(x, down=down, padding=pad.fir))
        return conv(fir(x, padding=pad.fir), stride=down)       # blur, then strided convolution (:119-122)

    if up > 1 and down == 1 and pointwise:  # convolve the smaller image, interpolate afterwards (:113-116)
        return fir(conv(x), up=up, padding=pad.fir, gain=up ** 2)

    if up > 1:                              # transposed strided convolution, then blur (:125-142)
        pad.shift(-(kw - 1), -(kw - up), -(kh - 1), -(kh - up))
        pxt = max(min(-pad.x0, -pad.x1), 0)
        pyt = max(min(-pad.y0, -pad.y1), 0)
        x = _conv2d_wrapper(x=x, w=_transposed_weight(w, groups), stride=up, padding=[pyt, pxt], groups=groups, transpose=True,
                            flip_weight=(not flip_weight), w_scale=w_scale)
        x = fir(x, padding=pad.shift(pxt, pxt, pyt, pyt).fir, gain=up ** 2)
        return fir(x, down=down) if down > 1 else x

    if pad.symmetric:                       # no resampling: plain convolution (:145-147)
        return conv(x, padding=pad.conv)

    # anything else (:150-154): pad with upfirdn2d, convolve without padding
    return conv(upfirdn2d.upfirdn2d(x=x, f=None, up=up, padding=pad.fir, gain=up ** 2, flip_filter=flip_filter))
