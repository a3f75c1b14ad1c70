"""conv2d / conv_transpose2d with arbitrary-order gradients, on the B200 tensor cores.

Drop-in for the reference's torch_utils/ops/conv2d_gradfix.py: same `conv2d`, `conv_transpose2d`,
`no_weight_gradients`, `enabled`, `weight_gradients_disabled`.  Where the reference wraps cuDNN
(conv2d_gradfix.py:112-114,143-145), this module runs the implicit-GEMM tcgen05 kernel
(csrc/conv_igemm.cu via `pgpp_conv2d_igemm`) for the forward and data-gradient convolutions.  The
autograd structure is the reference's (conv2d_gradfix.py:95-165): the data gradient of a convolution
is the opposite-transposed convolution and is itself differentiable, so R1's double backward works.

Switches
  enabled                    True: CUDA tensors take the sm_100a kernel (no fallback: unsupported
                             configurations raise).  False: plain torch.nn.functional (library) calls.
  weight_gradients_disabled  as in the reference (set by `no_weight_gradients()`).
  fp32_precision             how float32 tensors are fed to the bf16 tensor cores:
                             'bf16x3' 6 products of 3-term bf16 splits (~fp32 accuracy, rel 1e-6)
                             'bf16x2' 3 products of 2-term splits (rel ~1e-5; default, within the 1e-4 bar)
                             'bf16'   1 product (rel ~3e-3; what bf16/fp16 tensors always use)
                             'fp8'    opt-in, inference only: e4m3 operands on the kind::f8f6f4 MMA (activations at unit
                                      scale, saturating at +-448; weights with one fp32 scale per GEMM column), ~3.7e-2
                                      rel-L2 per layer.  A forward that autograd would record raises NotImplementedError.

The weight gradient (conv2d_gradfix.py:135-142) is the split-K tcgen05 GEMM over the pixels of
csrc/conv_wgrad.cu (`pgpp_conv2d_wgrad`); no library convolution is called anywhere on the path.
"""
import contextlib
import ctypes
import os
import threading
import weakref

import torch

from .. import custom_ops

enabled = True                      # the reference defaults to False and train.py flips it; here the kernel IS the path
weight_gradients_disabled = False
fp32_precision = 'bf16x2'
direct_few_tap_convs = os.environ.get('PGPP_NO_DIRECT_CONV') is None    # C*kh*kw <= 16 convs on the exact-fp32 direct kernel
# Training path: the forward pass keeps the packed (operand-format) copy of its input for the weight-gradient GEMM, and a plain
# backward pass (no create_graph) packs grad_output ONCE for both the data-gradient and the weight-gradient kernels instead of going
# through two more autograd Functions that each re-pack from NCHW.  Costs one operand-format copy per saved activation (the same
# bytes as the fp32 tensor in the bf16x2 mode) - sized for 180 GB of HBM3e.  False: re-pack in backward (round-1 behaviour).
keep_packed_operands = True

_PRODUCTS = {'bf16': (1, 1), 'bf16x2': (3, 2), 'bf16x3': (6, 3), 'f16': (1, 1), 'fp8': (1, 1)}    # name -> (MMA products, operand parts)
E4M3 = torch.float8_e4m3fn     # element type of the fp8 operand format
_ACT_IDX = {'linear': 1, 'relu': 2, 'lrelu': 3, 'tanh': 4, 'sigmoid': 5, 'elu': 6, 'selu': 7, 'softplus': 8, 'swish': 9}
_plugin = None
trace = None        # set to a list to record (label, algorithmic FLOPs, start event, end event) per igemm launch (bench.py roofline)


@contextlib.contextmanager
def no_weight_gradients():
    global weight_gradients_disabled
    old = weight_gradients_disabled
    weight_gradients_disabled = True
    yield
    weight_gradients_disabled = old


def _init():
    global _plugin
    if _plugin is None:
        _plugin = custom_ops.get_plugin('conv2d_plugin')
    return True


def _should_use_custom_op(input):
    assert isinstance(input, torch.Tensor)
    return enabled and input.device.type == 'cuda'


def _tuple_of_ints(xs, ndim):
    xs = tuple(xs) if isinstance(xs, (tuple, list)) else (xs,) * ndim
    assert len(xs) == ndim
    assert all(isinstance(x, int) for x in xs)
    return xs


def precision_for(dtype):
    """float32 / float64 tensors: the error-compensated bf16 split selected by `fp32_precision`; float16 tensors (the mixed-precision
    blocks of the discriminator, networks.py:634,647): native fp16 operands on the f16 tensor-core path, as cuDNN does for the
    reference; bfloat16 tensors: native bf16."""
    if dtype in (torch.float32, torch.float64):
        return fp32_precision
    return 'f16' if dtype == torch.float16 else 'bf16'


def check_fp8_forward_only(*tensors):
    """the fp8 precision is inference only: a float32 forward that autograd would record raises"""
    if (fp32_precision == 'fp8' and torch.is_grad_enabled() and
            any(t is not None and t.dtype in (torch.float32, torch.float64) and t.requires_grad for t in tensors)):
        raise NotImplementedError("fp32_precision = 'fp8' is an inference-only mode (no gradients); run the forward under torch.no_grad() "
                                  "or select 'bf16x3' / 'bf16x2' / 'bf16' for training")


# ------------------------------------------------------------------------------------------------
# operand packing (host logic; the packed weights are cached per parameter version)

def _round_up(v, m):
    return (v + m - 1) // m * m


def _split_bf16(t, parts):
    """[parts, ...] bf16 expansion of a float32 tensor: part p = bf16(t - sum of earlier parts)."""
    out = []
    rem = t.to(torch.float32)
    for _ in range(parts):
        q = rem.to(torch.bfloat16)
        out.append(q)
        rem = rem - q.to(torch.float32)
    return torch.stack(out)


class PackedWeights:
    """[parts, taps, o_rows, c_pad] bf16, K-major rows, ready for the TMA weight map.  e4m3: ONE part of e4m3 bytes with the column
    scales in `wscale` float32 [o_rows] (the weights of GEMM column g are data * wscale[g])."""
    __slots__ = ('data', 'master', 'kh', 'kw', 'o', 'phases', 'phase_stride', 'o_rows', 'c_pad', 'c_in', 'parts', 'pad_y', 'pad_x', 'im2col', 'f16',
                 'e4m3', 'wscale', 'e4m3_twin')


def e4m3_weights(pw):
    """the e4m3 form of bf16-packed weights (quantized from their float32 master rows, made once per PackedWeights): what an fp8 launch
    uses when a caller packed its weights for the bf16 formats (the generator's packers)"""
    if getattr(pw, 'e4m3', False):
        return pw
    twin = getattr(pw, 'e4m3_twin', None)
    if twin is None:
        assert pw.master is not None, 'fp16-packed weights have no float32 master rows'
        _init()
        data, ws = _plugin.quantize_weights_e4m3(pw.master.reshape(-1, pw.o_rows, pw.c_pad))
        twin = PackedWeights()
        for k in PackedWeights.__slots__:
            if k != 'e4m3_twin':
                setattr(twin, k, getattr(pw, k, None))
        twin.data, twin.wscale, twin.parts, twin.e4m3, twin.f16, twin.e4m3_twin = data[0], ws[0], 1, True, False, None
        pw.e4m3_twin = twin
    return twin


def e4m3_operand(x):
    """e4m3 copy of a one-part bf16 PackedAct (the hand-over format of the generator's route, which stays bf16 across its FIR, copy, mix and
    thin-conv kernels): the explicit bf16 -> e4m3 edge in front of an fp8 launch, one pgpp_pack_activations_e4m3 pass over the channel slice"""
    assert x.data.dtype == torch.bfloat16 and x.data.shape[0] == 1, 'the fp8 precision converts one-part bf16 operands only'
    _init()
    src = x.data[0, :, :, :, x.c_off:x.c_off + x.c].permute(0, 3, 1, 2)
    out = PackedAct(_plugin.pack_activations(src, None, _round_up(x.c, 64), 1, e4m3=True), x.c, 0, logical_hw=x.logical_hw)
    out.im2col = x.im2col
    return out


class PackedAct:
    """Activations in the tensor-core operand format: data [parts, N, H, W, c_total] bf16 (fp8 precision: one part of e4m3,
    dtype float8_e4m3fn), channels innermost; the
    logical tensor is channels [c_off, c_off + c) of every pixel.  Convolutions can write this format directly from
    their epilogue (`out_packed=`) and read it without a packing pass."""
    __slots__ = ('data', 'c', 'c_off', 'logical_hw', 'im2col')

    def __init__(self, data, c, c_off=0, logical_hw=None):
        self.data, self.c, self.c_off = data, c, c_off
        self.logical_hw = logical_hw        # (H, W) of the source image for row-group im2col operands (data has H + pad_y rows)
        self.im2col = None                  # im2col parameters when this operand was kept for the weight gradient (_forward_conv)

    @staticmethod
    def empty(n, h, w, c_total, parts, device, dtype=torch.bfloat16):
        """buffer with c_total rounded up to whole 64-channel swizzle rows; padding channels are zeroed (they meet zero weights,
        but must not hold NaN/Inf bit patterns)"""
        c_alloc = _round_up(c_total, 64)
        if c_alloc == c_total:
            return torch.empty([parts, n, h, w, c_alloc], dtype=dtype, device=device)
        return torch.zeros([parts, n, h, w, c_alloc], dtype=dtype, device=device)

    @property
    def shape(self):
        return (self.data.shape[1], self.c, self.data.shape[2], self.data.shape[3])

    @property
    def device(self):
        return self.data.device

    def view(self, c, c_off):
        return PackedAct(self.data, c, c_off)

    def to_nchw(self, dtype=torch.float32):
        """debug / test helper: sum of the parts as a [N, C, H, W] tensor"""
        v = self.data[:, :, :, :, self.c_off:self.c_off + self.c].to(torch.float32).sum(0)
        return v.permute(0, 3, 1, 2).contiguous().to(dtype)


def direct_conv_ok(weight, act='linear'):
    """few-tap convolutions (C*kh*kw <= 16, odd filter, 'same' padding) take the exact-fp32 direct kernel instead of being
    expanded to 64-channel tensor-core operands"""
    o, ic, kh, kw = weight.shape
    if not direct_few_tap_convs:
        return False
    return ic * kh * kw <= 16 and kh % 2 == 1 and kw in (1, 3) and act in ('linear', 'relu', 'lrelu')


def direct_conv(x, weight, bias=None, *, wscale=1.0, act='linear', alpha=0.0, gain=1.0, clamp=-1.0, out_packed=None):
    """y = clamp(act(conv2d(x, weight * wscale, padding='same') + bias) * gain) on pgpp_conv2d_direct; `out_packed`: PackedAct view
    to receive the operand format instead of returning an NCHW tensor"""
    _init()
    if out_packed is not None:
        assert out_packed.c == weight.shape[0]
        _plugin.conv2d_direct(x, weight, bias, wscale, _ACT_IDX[act], alpha, gain, clamp, out_packed.data, out_packed.c_off)
        return out_packed
    return _plugin.conv2d_direct(x, weight, bias, wscale, _ACT_IDX[act], alpha, gain, clamp)


def choose_block_n(cols, m_tiles, sms=148):
    bn = 256
    while bn > 16 and bn // 2 >= cols:
        bn //= 2
    while bn > 32 and m_tiles * ((cols + bn - 1) // bn) < sms:
        bn //= 2
    return bn


def pack_weights(w_taps, o, phases, kh, kw, parts, pad_y, pad_x):
    """w_taps: float32 [taps, phases*o, I] -> PackedWeights.  GEMM column of (phase, oc) is phase*phase_stride + oc
    (phase_stride = o rounded up to 16 when phases == 4); rows are padded to a multiple of 256 or to the
    power-of-two >= cols, channels to a multiple of 64."""
    taps, _, ic = w_taps.shape
    phase_stride = _round_up(o, 16) if phases > 1 else o
    cols = phases * phase_stride
    c_pad = _round_up(ic, 64)      # whole 128-byte swizzle rows: every conv takes the kb = 64 path with the unrolled MMA issue loop
    o_rows = _round_up(cols, 256) if cols > 128 else max(16, 1 << (cols - 1).bit_length())
    buf = torch.zeros([taps, o_rows, c_pad], dtype=torch.float32, device=w_taps.device)
    buf[:, :cols].reshape(taps, phases, phase_stride, c_pad)[:, :, :o, :ic] = w_taps.reshape(taps, phases, o, ic)
    pw = PackedWeights()
    pw.data = _split_bf16(buf, parts).contiguous()
    pw.master = buf.reshape(taps * o_rows, c_pad)       # fp32 rows for the per-sample (style-modulated) weight route
    pw.c_in = ic
    pw.kh, pw.kw, pw.o, pw.phases, pw.o_rows, pw.c_pad, pw.parts = kh, kw, o, phases, o_rows, c_pad, parts
    pw.phase_stride = phase_stride
    pw.pad_y, pw.pad_x = pad_y, pad_x
    pw.im2col = None
    pw.f16 = False
    pw.e4m3, pw.wscale = False, None
    return pw


def weight_layout(o, ic, phases=1):
    """(phase_stride, cols, o_rows, c_pad) of the packed weight operand: GEMM column of (phase, oc) is phase * phase_stride + oc
    (phase_stride = o rounded up to 16 for the 4-phase up=2 form); rows are padded to a multiple of 256 or to the power of two
    >= cols (whole N tiles), channels to whole 128-byte swizzle rows."""
    phase_stride = _round_up(o, 16) if phases > 1 else o
    cols = phases * phase_stride
    o_rows = _round_up(cols, 256) if cols > 128 else max(16, 1 << (cols - 1).bit_length())
    return phase_stride, cols, o_rows, _round_up(ic, 64)


def pack_weights_native(weights, kh, kw, parts, pad_y, pad_x, *, transpose_io=False, flip=False, scale=1.0, up2_filter=None, flip_filter=False,
                        f16=False, e4m3=False):
    """PackedWeights from one weight tensor - or several stacked along the output channels (gamma | beta of a SPADE block) - in ONE
    kernel launch per tensor (pgpp_pack_weights): scale, flip, transposition, padding, bf16 split / fp16 copy, and with `up2_filter`
    the polyphase form of the up=2 layer.  No library op touches the weights.  e4m3: the float32 rows are quantized to e4m3 with one
    scale per GEMM column (pgpp_quantize_weights_e4m3)."""
    _init()
    weights = list(weights) if isinstance(weights, (list, tuple)) else [weights]
    dims = [(int(w.shape[1]), int(w.shape[0])) if transpose_io else (int(w.shape[0]), int(w.shape[1])) for w in weights]
    ic = dims[0][1]
    assert all(d[1] == ic for d in dims)
    o = sum(d[0] for d in dims)
    phases = 4 if up2_filter is not None else 1
    assert phases == 1 or len(weights) == 1
    phase_stride, cols, o_rows, c_pad = weight_layout(o, ic, phases)
    taps = 9 if phases > 1 else kh * kw
    dev = weights[0].device
    dt = torch.float16 if f16 else torch.bfloat16
    alloc = torch.zeros if o_rows != cols else torch.empty          # rows beyond the tensor must read as zero weights
    pw = PackedWeights()
    pw.data = None if e4m3 else alloc([parts, taps, o_rows, c_pad], dtype=dt, device=dev)
    master = None if f16 else alloc([taps, o_rows, c_pad], dtype=torch.float32, device=dev)
    o_off = 0
    for w, (wo, _) in zip(weights, dims):
        _plugin.pack_weights(w, pw.data, master, transpose_io=transpose_io, flip=flip, scale=scale, phases=phases, phase_stride=phase_stride,
                             fir=up2_filter, flip_filter=flip_filter, parts=parts, f16=f16, o_off=o_off)
        o_off += wo
    pw.e4m3, pw.wscale = bool(e4m3), None
    if e4m3:
        assert parts == 1 and not f16
        data, ws = _plugin.quantize_weights_e4m3(master)
        pw.data, pw.wscale = data[0], ws[0]
    pw.master = None if master is None else master.reshape(taps * o_rows, c_pad)
    pw.c_in = ic
    pw.kh, pw.kw, pw.o, pw.phases, pw.o_rows, pw.c_pad, pw.parts = (3, 3, o, 4, o_rows, c_pad, parts) if phases > 1 else (kh, kw, o, 1, o_rows, c_pad, parts)
    pw.phase_stride = phase_stride
    pw.pad_y, pw.pad_x = pad_y, pad_x
    pw.im2col = None
    pw.f16 = bool(f16)
    return pw


_weight_cache = dict()      # (id(tensor), tag) -> (weakref(tensor), (data_ptr, _version, ...), None, packed); one entry per (parameter, tag)
_weight_cache_lock = threading.RLock()     # re-entrant: a weakref callback may fire while the lock is held


def _cached(key_tensor, tag, builder, also=()):
    """Packed weights per leaf tensor (Parameter / buffer) and `tag`.  An entry is valid while the SAME tensor object still owns
    the SAME storage address at the SAME `_version` (optimizer steps bump the version; `module.to()` / `param.data = ...` change
    the address), so a recycled address or a new version rebuilds and REPLACES the entry - nothing stale is returned and nothing
    piles up.  Temporaries (anything with a grad_fn, e.g. `self.weight * self.weight_gain` on the autograd path) are never
    cached: the entry could never hit again and would pin the temporary and its packed copies.
    `also`: further tensors the packed copy is built from (the second weight of a merged GEMM, the FIR filter)."""
    if key_tensor.grad_fn is not None or any(t.grad_fn is not None for t in also):
        return builder()
    key = (id(key_tensor), tag)
    stamp = (key_tensor.data_ptr(), key_tensor._version) + tuple(v for t in also for v in (id(t), t.data_ptr(), t._version))
    with _weight_cache_lock:
        hit = _weight_cache.get(key)
    if hit is not None and hit[0]() is key_tensor and hit[1] == stamp:
        return hit[3]
    value = builder()

    def _drop(_ref, key=key):
        with _weight_cache_lock:
            cur = _weight_cache.get(key)
            if cur is not None and cur[0] is _ref:
                del _weight_cache[key]
    with _weight_cache_lock:
        _weight_cache[key] = (weakref.ref(key_tensor, _drop), stamp, None, value)
    return value


def im2col_rows(ic, kh, kw):
    """rows per im2col group (0 = not worthwhile): r*kw*ic <= 64 with r >= min(kh, 3)"""
    if kh * kw == 1 or ic * kw > 21:
        return 0
    r = min(kh, 64 // (ic * kw))
    return r if (kh - 1) // r * r <= 6 else 0


def packed_plain(weight, flip_weight, parts, pad_y, pad_x, transpose_io=False, scale=1.0, allow_im2col=False, f16=False, e4m3=False):
    """weight [O, I, kh, kw] used as a correlation kernel (flip_weight=True, F.conv2d semantics) or a true
    convolution kernel (flip_weight=False).  transpose_io: weight is [I, O, kh, kw] (conv_transpose2d layout).
    scale: constant folded into the packed copy (the layers' runtime weight_gain, networks.py:155,169)."""
    def build():
        o, ic, kh, kw = (weight.shape[1], weight.shape[0], *weight.shape[2:]) if transpose_io else weight.shape
        r = im2col_rows(ic, kh, kw) if allow_im2col else 0
        if not r:
            return pack_weights_native(weight, kh, kw, parts, pad_y, pad_x, transpose_io=transpose_io, flip=not flip_weight, scale=float(scale),
                                       f16=f16, e4m3=e4m3)
        assert not f16 and not e4m3
        w = weight.detach().to(torch.float32) * float(scale)
        if transpose_io:
            w = w.transpose(0, 1)
        if not flip_weight:
            w = w.flip([2, 3])
        if True:
            # row-group im2col operand (pgpp_pack_im2col): channel (ry*kw + kx)*ic + c of vertical tap group t holds w[o, c, t*r + ry, kx]
            groups = -(-kh // r)
            wp = torch.zeros([groups, o, r, kw, ic], dtype=torch.float32, device=w.device)
            for t in range(groups):
                rows = min(r, kh - t * r)
                wp[t, :, :rows] = w[:, :, t * r:t * r + rows, :].permute(0, 2, 3, 1)
            pw = pack_weights(wp.reshape(groups, o, r * kw * ic), o, 1, groups, 1, parts, 0, 0)
            pw.im2col = dict(r=r, kw=kw, kh=kh, pad_x=pad_x, pad_y=pad_y)
            return pw
    return _cached(weight, ('plain', bool(flip_weight), parts, pad_y, pad_x, bool(transpose_io), float(scale), bool(allow_im2col), bool(f16)) +
                   (('e4m3',) if e4m3 else ()), build)


_UP2_TAPS = ((2, 0), (1,))      # phase r of a stride-2 transposed 3-tap convolution: T[2j + r] = sum_t x[j + t - pad_r] * w[_UP2_TAPS[r][t]], pad_0 = 1, pad_1 = 0


def packed_up2_phase(weight, ry, rx, flip_weight, parts, e4m3=False):
    """Phase (ry, rx) of `conv_transpose2d(x, w', stride=2)` for a 3 x 3 kernel as a correlation over the INPUT grid (w' = the kernel as
    conv_transpose2d sees it, conv2d_resample.py:131-132):  T[2j + ry, 2i + rx] = sum_{ty, tx} x[j + ty - (1 - ry), i + tx - (1 - rx)] * w'[KY[ty], KX[tx]]
    with KY = (2, 0) for ry = 0 and (1,) for ry = 1: 2 x 2, 2 x 1, 1 x 2 and 1 x 1 taps - the nine taps of the kernel, each used once."""
    def build():
        assert tuple(weight.shape[2:]) == (3, 3)
        w = weight.detach()
        if flip_weight:
            w = w.flip([2, 3])
        ky = torch.tensor(_UP2_TAPS[ry], device=w.device)
        kx = torch.tensor(_UP2_TAPS[rx], device=w.device)
        sub = w.index_select(2, ky).index_select(3, kx).contiguous()
        return pack_weights_native(sub, len(_UP2_TAPS[ry]), len(_UP2_TAPS[rx]), parts, 1 - ry, 1 - rx, e4m3=e4m3)
    return _cached(weight, ('up2_phase', ry, rx, bool(flip_weight), parts) + (('e4m3',) if e4m3 else ()), build)


def packed_up2_taps4(weight, flip_weight, parts, e4m3=False):
    """`conv_transpose2d(x, w', stride=2)` for a 3 x 3 kernel as ONE 2 x 2 correlation over the input grid with 4 * O GEMM columns (phase-major,
    phase = 2 ry + rx writes T[2j + ry, 2i + rx]): tap (dy, dx) of the 2 x 2 window (padding 1) carries w'[KY, KX] for the phases that use that
    input offset and zeros for the others - 16 instead of the algorithmic 9 MACs per input pixel and (output, input) channel pair (the polyphase
    form with the blur folded in needs 36), but the input is read once and the four phases leave in one launch."""
    def build():
        assert tuple(weight.shape[2:]) == (3, 3)
        w = weight.detach().to(torch.float32)
        if flip_weight:
            w = w.flip([2, 3])
        o, ic = w.shape[:2]
        assert o % 16 == 0
        w4 = torch.zeros([4, o, ic, 2, 2], dtype=torch.float32, device=w.device)
        for ry in (0, 1):
            for rx in (0, 1):
                for ty, ky in enumerate(_UP2_TAPS[ry]):
                    for tx, kx in enumerate(_UP2_TAPS[rx]):
                        w4[2 * ry + rx, :, :, ty + ry, tx + rx] = w[:, :, ky, kx]      # odd phases use only the window offset 1 (the pixel itself)
        pw = pack_weights_native(w4.reshape(4 * o, ic, 2, 2), 2, 2, parts, 1, 1, e4m3=e4m3)
        pw.phases, pw.o, pw.phase_stride = 4, o, o
        return pw
    return _cached(weight, ('up2_taps4', bool(flip_weight), parts) + (('e4m3',) if e4m3 else ()), build)


def up2_modconv_packed(xp, weight, styles, dcoef, f, flip_weight, out_packed, *, noise=None, bias=None, act='linear', alpha=0.0, gain=1.0, clamp=-1.0,
                       taps4=False):
    """The StyleGAN2 up = 2 modulated layer at the algorithmic MAC count, operand format in and out: the transposed convolution as four
    per-phase implicit GEMMs (demodulation in their epilogue) writing the (2H + 1) x (2W + 1) intermediate in the operand format, then ONE
    pass `pgpp_fir_packed_act` = 4 x 4 blur (gain 4) + noise + bias + activation + clamp into `out_packed` (None: a float32 NCHW tensor is returned).  Against the polyphase form
    (`packed_up2`, one launch at 4x the MACs) this wins on the tensor-bound layers (C >= 128)."""
    _init()
    n, _, h, w = xp.shape
    parts = xp.data.shape[0]
    e4m3 = xp.data.dtype == E4M3        # e4m3 GEMMs; the intermediate and the blur pass stay in bf16 (one part)
    o = weight.shape[0]
    if taps4:
        # `taps4`: the four phases as ONE 2 x 2 GEMM with 4 * O columns (16 / 9 of the algorithmic MACs, the input read once) - for the layers
        # where four passes over the input cost more than the extra MACs.  Its grid is (H + 1) x (W + 1), so the intermediate has 2H + 2 rows, the
        # last one zero (x[H] is outside the image): it stands in for the blur's bottom / right padding.
        t = PackedAct(PackedAct.empty(n, 2 * h + 2, 2 * w + 2, o, parts, xp.device), o)
        igemm_conv(xp, packed_up2_taps4(weight, flip_weight, parts, e4m3), scale=styles, dcoef=dcoef, out_hw=(h + 1, w + 1), out_packed=t)
        pad = (1, 0, 1, 0)
    else:
        t = PackedAct(PackedAct.empty(n, 2 * h + 1, 2 * w + 1, o, parts, xp.device), o)
        for ry in (0, 1):
            for rx in (0, 1):
                pw = packed_up2_phase(weight, ry, rx, flip_weight, parts, e4m3)
                igemm_conv(xp, pw, scale=styles, dcoef=dcoef, out_hw=(h + 1 - ry, w + 1 - rx), out_packed=t, out_phase=(ry, rx))
        pad = (1, 1, 1, 1)
    taps, fw, fh = host_filter(f)
    if out_packed is None:          # float32 NCHW result
        y = torch.empty([n, o, 2 * h, 2 * w], dtype=torch.float32, device=xp.device)
        return _plugin.fir_packed_act(t.data, o, 0, taps, fw, fh, *pad, False, 4.0, noise, bias, _ACT_IDX[act], alpha, gain, clamp, None, dst_nchw=y)
    _plugin.fir_packed_act(t.data, o, 0, taps, fw, fh, *pad, False, 4.0, noise, bias, _ACT_IDX[act], alpha, gain, clamp,
                           out_packed.data, dst_c_off=out_packed.c_off)
    return out_packed


def packed_up2(weight, f, flip_weight, flip_filter, parts, e4m3=False):
    """Polyphase form of `conv_transpose2d(stride=2)` followed by the 4x4 FIR with gain 4
    (conv2d_resample.py:125-139, the StyleGAN2 up=2 layer): for output pixel (2y+py, 2x+px)

        out = sum_{a,b in 0..2} x[y+a-1, x+b-1] * Wp[py,px][o,i,a,b]
        Wp[py,px][.,.,a,b] = 4 * sum_{fy,ky: py+fy-1-ky = 2(a-1)} sum_{fx,kx: px+fx-1-kx = 2(b-1)} w'[ky,kx] * k[fy,fx]

    with w' the kernel as conv_transpose2d sees it and k the (flipped) FIR.  One 3x3 GEMM with 4*O columns
    replaces the transposed convolution, its (2H+1)^2 intermediate and the blur pass."""
    def build():
        assert tuple(weight.shape[2:]) == (3, 3) and tuple(f.shape) == (4, 4) and f.dtype == torch.float32
        return pack_weights_native(weight, 3, 3, parts, 1, 1, flip=bool(flip_weight), up2_filter=f, flip_filter=bool(flip_filter), e4m3=e4m3)
    return _cached(weight, ('up2', bool(flip_weight), bool(flip_filter), parts) + (('e4m3',) if e4m3 else ()), build, also=(f,))


_host_filter_cache = dict()     # id(filter tensor) -> (weakref, (data_ptr, _version), (taps, fw, fh))


def host_filter(f):
    """(taps, fw, fh) of a FIR filter tensor as host floats (one device -> host copy per filter tensor, first use only); a 1-D
    filter is the separable pair, i.e. its outer product (upfirdn2d.py:103-106)"""
    key = id(f)
    hit = _host_filter_cache.get(key)
    if hit is not None and hit[0]() is f and hit[1] == (f.data_ptr(), f._version):
        return hit[2]
    ff = f.detach().to(torch.float32).cpu()
    if ff.ndim == 1:
        ff = ff.ger(ff)
    assert ff.ndim == 2 and ff.shape[0] <= 4 and ff.shape[1] <= 4, 'the operand-format FIR takes filters of at most 4 x 4 taps'
    val = ([float(v) for v in ff.reshape(-1)], int(ff.shape[1]), int(ff.shape[0]))
    _host_filter_cache[key] = (weakref.ref(f, lambda _r, key=key: _host_filter_cache.pop(key, None)), (f.data_ptr(), f._version), val)
    return val


def fir_packed(xp, f, down=1, padding=(0, 0, 0, 0), flip_filter=False, gain=1.0, out=None):
    """`upfirdn2d(x, f, down=down, padding=[padx0, padx1, pady0, pady1], flip_filter=..., gain=...)` on a PackedAct, result as a
    PackedAct (`out`: PackedAct view to write into, else a new buffer): the blur / decimation in front of a down-sampling convolution
    (conv2d_resample.py:107-110, 119-122) without leaving the operand format.  f=None copies the channel slice."""
    _init()
    taps, fw, fh = (None, 1, 1) if f is None else host_filter(f)
    px0, px1, py0, py1 = (int(v) for v in padding)
    if out is None:
        data = _plugin.fir_packed(xp.data, xp.c, xp.c_off, taps, fw, fh, down, px0, px1, py0, py1, flip_filter, gain)
        return PackedAct(data, xp.c)
    assert out.c == xp.c
    _plugin.fir_packed(xp.data, xp.c, xp.c_off, taps, fw, fh, down, px0, px1, py0, py1, flip_filter, gain, dst=out.data, dst_c_off=out.c_off)
    return out


# ------------------------------------------------------------------------------------------------
# the kernel launch

def igemm_conv(x, pw, *, scale=None, stride=1, out_hw=None, dcoef=None, noise=None, bias=None, act='linear',
               alpha=0.0, gain=1.0, clamp=-1.0, out=None, out_dtype=None, accumulate=False, precision=None,
               memory_format=None, out_packed=None, spade=None, instnorm_eps=None, out_phase=None):
    """Run one fused convolution.
    x          [N, I, H, W] tensor (any float dtype / layout; packed here, `scale` [N, I] = style modulation folded into the
               packing pass) or a PackedAct (no packing pass; `scale` is then folded into per-sample weights).
    out_packed None -> returns a [N, O, out_h, out_w] tensor (`out` / `out_dtype` / `memory_format` as given);
               PackedAct view -> the epilogue writes the bf16 operand format of the next conv into that channel slice.
    spade      (x_norm [N, C, H, W] float32, mean [N, C], rstd [N, C], pre_gain): the GEMM's O = 2C columns are gamma | beta and the
               epilogue writes pre_act((x_norm - mean) * rstd * (1 + gamma) + beta) into `out_packed` (C channels).
    out_phase  (ry, rx) with `out_packed` a PackedAct over a (2 * conv_h' + 1) x (2 * conv_w' + 1) grid: the result pixel (j, i) is written to
               (2 j + ry, 2 i + rx) of it - one phase of a stride-2 transposed convolution (conv2d_resample.py:125-139) at 1x its MACs.
    instnorm_eps  not None -> returns (y, mean [N, O], rstd [N, O]): the instance-norm statistics of the float32 NCHW result
               (torch.var_mean(y, (2, 3), unbiased=False), rstd = rsqrt(var + eps)), from partial sums the epilogue leaves per warp and a
               small float64 merge kernel - no second pass over y.  Launches that cannot produce them fall back to torch.var_mean."""
    _init()
    n, ic, h, w = x.shape
    im = pw.im2col
    if im is not None:
        assert stride == 1 and out_hw is None
        if isinstance(x, PackedAct):
            src_h, src_w = x.logical_hw
        else:
            src_h, src_w = h, w
        out_hw = (src_h + 2 * im['pad_y'] - im['kh'] + 1, src_w + 2 * im['pad_x'] - im['kw'] + 1)
    src_dtype = torch.float32 if isinstance(x, PackedAct) else x.dtype
    precision = precision or precision_for(src_dtype)
    products, parts = _PRODUCTS[precision]
    f16 = precision == 'f16'
    e4m3 = precision == 'fp8'
    esize = 1 if e4m3 else 2        # bytes per operand element
    converted = False
    if e4m3:        # operands packed for the bf16 formats take the explicit bf16 -> e4m3 edge
        pw = e4m3_weights(pw)
        if isinstance(x, PackedAct) and x.data.dtype != E4M3:
            x, converted = e4m3_operand(x), True
    assert pw.parts >= parts, 'weights were packed with fewer parts than the requested precision needs'
    assert bool(pw.f16) == f16, 'fp16 operands need fp16-packed weights (and only they)'
    assert bool(getattr(pw, 'e4m3', False)) == e4m3, 'e4m3 operands need e4m3-packed weights (and only they)'
    d = custom_ops.ConvDesc()
    keep = []
    if isinstance(x, PackedAct):
        assert x.data.shape[0] >= parts and x.c_off % (16 if e4m3 else 8) == 0
        assert (x.data.dtype == E4M3) == e4m3, 'the fp8 precision takes e4m3 operands (and only it)'
        assert pw.c_pad <= x.data.shape[4] - x.c_off, 'packed activations have fewer channels than the weights expect'
        d.act = x.data.data_ptr() + esize * x.c_off
        d.a_parts = x.data.shape[0]
        d.act_pixel_stride = x.data.shape[4]
        device = x.data.device
        if scale is not None and e4m3:      # per-sample weights: e4m3 bytes and column scales of master * styles
            wdata, wsc = _plugin.quantize_weights_e4m3(pw.master.reshape(-1, pw.o_rows, pw.c_pad), scale)
            keep += [wdata, wsc]
            d.wgt = wdata.data_ptr(); d.b_parts = 1; d.wgt_per_sample = 1; d.wscale = wsc.data_ptr()
        elif scale is not None:       # style modulation folded into per-sample weights (needs >= 128 pixels per sample)
            wdata = _plugin.modulate_weights(pw.master, scale, parts)
            keep.append(wdata)
            d.wgt = wdata.data_ptr(); d.b_parts = parts; d.wgt_per_sample = 1
        else:
            d.wgt = pw.data.data_ptr(); d.b_parts = pw.data.shape[0]
    else:
        if im is not None:
            x_packed = _plugin.pack_im2col(x, scale, im['kw'], im['r'], im['pad_x'], im['pad_y'], parts)
            h = x_packed.shape[2]
            if e4m3:        # the row-group im2col operand is packed in bf16, then takes the bf16 -> e4m3 edge
                x_packed = e4m3_operand(PackedAct(x_packed, x_packed.shape[4])).data
        else:
            x_packed = _plugin.pack_activations(x, scale, pw.c_pad, parts, f16=f16, e4m3=e4m3)
        keep.append(x_packed)
        d.act = x_packed.data_ptr(); d.a_parts = parts
        d.wgt = pw.data.data_ptr(); d.b_parts = pw.data.shape[0]
        device = x.device
    if e4m3:
        d.operand_e4m3 = 1
        if not d.wgt_per_sample:
            d.wscale = pw.wscale.data_ptr()
    up = 2 if pw.phases == 4 else 1
    if out_hw is None:
        conv_h = (h + 2 * pw.pad_y - pw.kh) // stride + 1
        conv_w = (w + 2 * pw.pad_x - pw.kw) // stride + 1
    else:
        conv_h, conv_w = out_hw
    out_h, out_w = conv_h * up, conv_w * up
    if out_packed is not None and out_phase is not None:
        ry, rx = out_phase
        th_, tw_ = int(out_packed.data.shape[2]), int(out_packed.data.shape[3])
        assert out_packed.data.shape[1] == n and 2 * (out_h - 1) + ry < th_ and 2 * (out_w - 1) + rx < tw_ and out_packed.c == pw.o
        assert pw.o % 16 == 0 and out_packed.c_off % 8 == 0 and up == 1 and spade is None
        c_total = out_packed.data.shape[4]
        d.out = out_packed.data.data_ptr() + out_packed.data.element_size() * (out_packed.c_off + (ry * tw_ + rx) * c_total)
        d.out_dtype = custom_ops.dtype_code(out_packed.data.dtype)
        d.out_stride = (ctypes.c_int64 * 4)(th_ * tw_ * c_total, 1, 2 * tw_ * c_total, 2 * c_total)
        d.out_parts = out_packed.data.shape[0]
        d.out_part_stride = out_packed.data[0].numel()
        result = out_packed
    elif out_packed is not None:
        assert tuple(out_packed.data.shape[1:4]) == (n, out_h, out_w) and out_packed.c == (pw.o // 2 if spade is not None else pw.o)
        assert pw.o % 16 == 0 and out_packed.c_off % 8 == 0
        c_total = out_packed.data.shape[4]
        d.out = out_packed.data.data_ptr() + out_packed.data.element_size() * out_packed.c_off
        d.out_dtype = custom_ops.dtype_code(out_packed.data.dtype)      # bf16 parts, or e4m3 from e4m3 operands
        d.out_stride = (ctypes.c_int64 * 4)(out_h * out_w * c_total, 1, out_w * c_total, c_total)
        d.out_parts = out_packed.data.shape[0]
        d.out_part_stride = out_packed.data[0].numel()
        result = out_packed
    else:
        want_f64 = out is None and out_dtype is None and src_dtype == torch.float64      # computed in the fp32-parity mode, returned as float64
        if out is None:
            out_dtype = out_dtype or (src_dtype if src_dtype != torch.float64 else torch.float32)
            if memory_format is None:
                cl = (not isinstance(x, PackedAct)) and x.stride(1) == 1 and ic > 1
                memory_format = torch.channels_last if cl else torch.contiguous_format
            out = torch.empty([n, pw.o, out_h, out_w], dtype=out_dtype, device=device, memory_format=memory_format)
        assert tuple(out.shape) == (n, pw.o, out_h, out_w)
        d.out = out.data_ptr(); d.out_dtype = custom_ops.dtype_code(out.dtype)
        d.out_stride = (ctypes.c_int64 * 4)(*out.stride())
        d.out_parts = 1
        result = out

    tw = min(128, 1 << (conv_w - 1).bit_length())
    th = min(128 // tw, 1 << (conv_h - 1).bit_length())
    tn = 128 // (tw * th)
    m_tiles = -(-conv_w // tw) * -(-conv_h // th) * -(-n // tn)
    block_n = choose_block_n(pw.phases * pw.phase_stride, m_tiles)
    while pw.o_rows % block_n:
        block_n //= 2
    if spade is not None:
        sx, smean, srstd, spre = spade
        assert out_packed is not None and pw.phases == 1 and pw.o % 32 == 0 and pw.o in (32, 64, 128, 256) and pw.o_rows % pw.o == 0
        assert sx.dtype == torch.float32 and sx.is_contiguous() and tuple(sx.shape) == (n, pw.o // 2, out_h, out_w)
        smean = smean.detach().to(torch.float32).reshape(n, pw.o // 2).contiguous()
        srstd = srstd.detach().to(torch.float32).reshape(n, pw.o // 2).contiguous()
        keep += [smean, srstd]
        block_n = pw.o          # gamma and beta of a channel must sit in the same accumulator tile
        d.spade_x = sx.data_ptr(); d.spade_mean = smean.data_ptr(); d.spade_rstd = srstd.data_ptr(); d.spade_pre_gain = float(spre)

    d.n, d.h, d.w, d.c_pad = n, h, w, pw.c_pad
    d.kh, d.kw, d.pad_y, d.pad_x, d.stride = pw.kh, pw.kw, pw.pad_y, pw.pad_x, stride
    d.dil_y = im['r'] if (im is not None and pw.kh > 1) else 1
    d.conv_h, d.conv_w = conv_h, conv_w
    d.o, d.phases, d.phase_stride, d.o_rows, d.block_n, d.products = pw.o, pw.phases, pw.phase_stride, pw.o_rows, block_n, products
    def fptr(t):
        if t is None:
            return None
        t = t.detach().to(torch.float32).contiguous()
        keep.append(t)
        return t.data_ptr()
    d.dcoef = fptr(dcoef)
    if noise is not None:
        nz = noise.detach().to(torch.float32)
        if nz.dim() == 4:       # [N, 1, H, W]
            nz = nz.reshape(nz.shape[0], out_h, out_w).contiguous()
            d.noise_stride_n = out_h * out_w if nz.shape[0] > 1 else 0
        else:
            nz = nz.reshape(out_h, out_w).contiguous()
            d.noise_stride_n = 0
        keep.append(nz)
        d.noise = nz.data_ptr()
    d.bias = fptr(bias)
    d.act_fn = _ACT_IDX[act]; d.alpha = float(alpha); d.gain = float(gain); d.clamp = float(clamp)
    d.out_h, d.out_w = out_h, out_w
    d.accumulate = int(bool(accumulate))
    d.operand_f16 = int(f16)
    stats_ws = None
    if instnorm_eps is not None:
        assert out_packed is None and spade is None
        rows = _plugin.conv2d_igemm_plan(d)['stats_rows'] if (result.dtype == torch.float32 and result.is_contiguous()) else 0
        if rows > 0:
            stats_ws = torch.empty([3, rows, pw.o], dtype=torch.float32, device=device)
            d.stats_ws = stats_ws.data_ptr()
    if trace is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _plugin.conv2d_igemm(d, device)
        e1.record()
        # algorithmic FLOPs (SURVEY 8d): 2*N*O*I*kh*kw*P; for the polyphase up=2 form the transposed conv's 9 taps per INPUT pixel
        real_ic, real_taps = (ic, 9 if pw.phases == 4 else pw.kh * pw.kw) if im is None else (pw.c_in // (im['r'] * im['kw']), im['kh'] * im['kw'])
        flops = 2.0 * n * pw.o * real_ic * real_taps * conv_h * conv_w
        kname = f'k{pw.kh}' if im is None else f"k{im['kh']}(im2col r{im['r']})"
        okind = ('spade' if spade is not None else 'packed' if out_packed is not None else 'nchw') + ('+acc' if accumulate else '')
        ikind = ('packed(bf16->e4m3)' if converted else 'packed') if isinstance(x, PackedAct) else 'tensor'
        elem = f'{precision}(e4m3)' if e4m3 else precision         # the operand element type that ran
        trace.append((f'igemm {real_ic}->{pw.o} {kname} {h}x{w}->{out_h}x{out_w} n{n} {elem} {ikind}->{okind}', flops, e0, e1))
    else:
        _plugin.conv2d_igemm(d, device)
    if out_packed is None and want_f64:
        result = result.to(torch.float64)       # the reference returns the input dtype (conv2d_gradfix.py:112-114)
    if instnorm_eps is not None:
        if stats_ws is not None:
            mean, rstd = _plugin.instnorm_finalize(stats_ws, n, instnorm_eps)
        else:
            var, mean = torch.var_mean(result.to(torch.float32), dim=(2, 3), unbiased=False)
            rstd = (var + instnorm_eps).rsqrt()
        return result, mean, rstd
    return result


# ------------------------------------------------------------------------------------------------
# public API

def _library_weight(input, weight, weight_scale):
    w = weight if weight_scale == 1.0 else weight * weight_scale
    return w if w.dtype == input.dtype else w.to(input.dtype)


FUSED_EPILOGUE_ACTS = ('linear', 'relu', 'lrelu')     # activations whose gradient needs the OUTPUT only (bias_act.py:24-34 `ref='y'` / '')


def conv2d(input, weight, bias=None, stride=1, padding=0, dilation=1, groups=1, weight_scale=1.0, epilogue=None):
    """`weight_scale` (extension to conv2d_gradfix.py:22-25): the result is conv2d(input, weight * weight_scale) with the constant folded
    into the packed copy of `weight` - pass the PARAMETER itself (float32 also for float16 inputs) instead of `weight * gain` and the
    packed copy is made once per optimizer step, not once per call.
    `epilogue` (extension, kernel path only): (act, alpha, gain, clamp) of the bias_act call that would follow - clamp(act(conv + bias) * gain)
    comes out of the convolution's epilogue instead of a second pass over the result; its gradient is bias_act's own gradient op on the
    saved output, so first and second order gradients are those of conv2d followed by bias_act."""
    if _should_use_custom_op(input):
        check_fp8_forward_only(input, weight, bias)
        if epilogue is not None:
            act, alpha, gain, clamp = epilogue
            assert act in FUSED_EPILOGUE_ACTS
            epilogue = (act, float(alpha), float(gain), float(clamp))
        return _conv2d_gradfix(transpose=False, weight_shape=weight.shape, stride=stride, padding=padding, output_padding=0,
                               dilation=dilation, groups=groups, weight_scale=float(weight_scale), epilogue=epilogue).apply(input, weight, bias)
    assert epilogue is None, 'epilogue= needs the kernel path'
    return torch.nn.functional.conv2d(input=input, weight=_library_weight(input, weight, weight_scale), bias=bias, stride=stride, padding=padding,
                                      dilation=dilation, groups=groups)


def conv_transpose2d(input, weight, bias=None, stride=1, padding=0, output_padding=0, groups=1, dilation=1, weight_scale=1.0):
    if _should_use_custom_op(input):
        check_fp8_forward_only(input, weight, bias)
        return _conv2d_gradfix(transpose=True, weight_shape=weight.shape, stride=stride, padding=padding,
                               output_padding=output_padding, groups=groups, dilation=dilation, weight_scale=float(weight_scale)).apply(input, weight, bias)
    return torch.nn.functional.conv_transpose2d(input=input, weight=_library_weight(input, weight, weight_scale), bias=bias, stride=stride,
                                                padding=padding, output_padding=output_padding, groups=groups, dilation=dilation)


def pack_operand(x, prec=None):
    """NCHW (or any-strided) tensor -> PackedAct in the operand format of `prec` (channels padded to whole 64-channel rows)"""
    _init()
    prec = prec or precision_for(x.dtype)
    data = _plugin.pack_activations(x, None, _round_up(x.shape[1], 64), _PRODUCTS[prec][1], f16=prec == 'f16', e4m3=prec == 'fp8')
    return PackedAct(data, x.shape[1])


def _im2col_plan(x, weight, stride, padding):
    """row-group im2col parameters for a few-channel convolution on an NCHW tensor (None: take the plain operand): C * kw <= 21, 'same' or any
    symmetric padding, stride 1, images of at least 8 x 16 - the 7 x 7 RGB stems and the 3 x 3 convolutions on 1..6-channel maps, whose
    64-channel operand rows would otherwise be 95 % padding"""
    if isinstance(x, PackedAct) or tuple(stride) != (1, 1) or x.dtype not in (torch.float32, torch.bfloat16):
        return None
    o, ic, kh, kw = weight.shape
    if x.shape[2] < 8 or x.shape[3] < 16 or o % 16 != 0:
        return None
    r = im2col_rows(ic, kh, kw)
    return dict(r=r, kh=kh, kw=kw, ic=ic, pad_y=int(padding[0]), pad_x=int(padding[1])) if r else None


def _weight_gradient_im2col(go, xim, weight_shape, im, precision, out_dtype):
    """dW of a convolution that ran on the row-group im2col operand `xim` ([parts, N, H + pad_y, W, 64]: channel (ry * kw + kx) * ic + c of row
    yy holds x[c, yy - pad_y + ry, x + kx - pad_x]): the weight gradient of the equivalent (groups x 1)-tap convolution with vertical tap spacing
    r, G[o, ch, g] = sum gy[o, y, x] * xim[y + g * r, x, ch], scattered back to [O, I, kh, kw] (ky = g * r + ry)."""
    o, ic, kh, kw = (int(v) for v in weight_shape)
    r = im['r']
    groups = -(-kh // r)
    g = weight_gradient(go, xim, (o, r * kw * ic, groups, 1), 1, (0, 0), False, precision=precision, out_dtype=torch.float32, dil_y=r)
    g = g.reshape(o, r, kw, ic, groups).permute(0, 3, 4, 1, 2).reshape(o, ic, groups * r, kw)[:, :, :kh]
    return g.contiguous().to(out_dtype)


def _forward_conv(x, weight, bias, stride, padding, keep=False, scale=1.0, epi=None):
    """F.conv2d(x, weight, bias, stride, padding) on the tensor cores.  x: tensor or PackedAct (then `keep` is moot).
    keep=True also returns the packed copy of x (for the weight gradient).  epi: dict(act, alpha, gain, clamp) applied by the epilogue."""
    epi = epi or {}
    src_dtype = (torch.float16 if x.data.dtype == torch.float16 else weight.dtype) if isinstance(x, PackedAct) else x.dtype   # f16 operands: fp16 layer
    prec = precision_for(src_dtype)
    im = _im2col_plan(x, weight, stride, padding) if prec not in ('f16', 'fp8') else None
    if im is not None:
        # few-channel convolution: all taps of r filter rows go into the channel dimension (pgpp_pack_im2col); the operand is kept for the
        # weight gradient, which runs on it too
        _init()
        parts = _PRODUCTS[prec][1]
        pw = packed_plain(weight, True, parts, padding[0], padding[1], scale=scale, allow_im2col=True)
        assert pw.im2col is not None
        xp = PackedAct(_plugin.pack_im2col(x, None, im['kw'], im['r'], im['pad_x'], im['pad_y'], parts), im['r'] * im['kw'] * im['ic'], 0,
                       logical_hw=(int(x.shape[2]), int(x.shape[3])))
        mf = torch.channels_last if (x.stride(1) == 1 and x.shape[1] > 1) else torch.contiguous_format
        y = igemm_conv(xp, pw, bias=bias, precision=prec, out_dtype=src_dtype, memory_format=mf, **epi)
        if keep:
            xp.im2col = im
            return y, xp
        return y
    pw = packed_plain(weight, True, _PRODUCTS[prec][1], padding[0], padding[1], f16=prec == 'f16', scale=scale, e4m3=prec == 'fp8')
    xp, mf = x, None
    if keep and not isinstance(x, PackedAct):
        mf = torch.channels_last if (x.stride(1) == 1 and x.shape[1] > 1) else torch.contiguous_format     # the output follows the input's layout
        xp = pack_operand(x, prec)
    y = igemm_conv(xp, pw, stride=stride[0], bias=bias, precision=prec, out_dtype=src_dtype if src_dtype != torch.float64 else None,
                   memory_format=mf, **epi)
    if src_dtype == torch.float64 and y.dtype != torch.float64:
        y = y.to(torch.float64)
    return (y, xp) if keep else y


FUSE_ACT_GRAD_PACK = True      # plain backward of a convolution with a fused bias_act: dy * act'(y) straight into the operand format (pgpp_pack_act_gradient)

TCONV_PHASES = True      # stride-2 transposed convolutions (the data gradient of every down-sampling convolution) as four per-phase convolutions of
                         # the un-stuffed input at 1x the MACs; False: zero insertion + one convolution over the 4x larger tensor (the round-1 form)


def tconv_stride2_phase_plan(kh, kw, padding):
    """Stride-2 transposed convolution as four stride-1 correlations (pure arithmetic, no tensors):
    y[i] = sum_{j, t: 2 j + t - p = i} x[j] * w[t].  Output phase r = i & 1 only sees the taps t = t0 + 2 m with t0 = (r + p) & 1, at inputs
    j = q + s - m (i = 2 q + r, s = (r + p - t0) / 2): a stride-1 correlation of x with the flipped sub-kernel w[t0::2], padding (T - 1) - s
    (may be negative = a crop), whose result is every second pixel of y.  -> one entry per (ry, rx):
    dict(ry, rx, t0y, t0x, ty, tx, pad_y, pad_x); ty == 0 or tx == 0: no tap reaches that phase (the output there is the bias)."""
    plan = []
    for ry in (0, 1):
        t0y = (ry + padding[0]) & 1
        ty = max(0, (kh - t0y + 1) // 2)
        for rx in (0, 1):
            t0x = (rx + padding[1]) & 1
            tx = max(0, (kw - t0x + 1) // 2)
            plan.append(dict(ry=ry, rx=rx, t0y=t0y, t0x=t0x, ty=ty, tx=tx,
                             pad_y=(ty - 1) - (ry + padding[0] - t0y) // 2, pad_x=(tx - 1) - (rx + padding[1] - t0x) // 2))
    return plan


def _conv_transpose_stride2_phases(x, weight, bias, padding, output_padding, scale):
    """F.conv_transpose2d(x, weight[I, O, kh, kw], stride=2, ...) by `tconv_stride2_phase_plan`: four launches on ONE packed copy of x, each
    writing a strided output view of the implicit GEMM, instead of a zero-insertion pass, a packing pass over the 4x larger tensor and a
    convolution that multiplies 75 % zeros."""
    _init()
    ic, oc, kh, kw = (int(v) for v in weight.shape)
    src_dtype = (torch.float16 if x.data.dtype == torch.float16 else weight.dtype) if isinstance(x, PackedAct) else x.dtype
    prec = precision_for(src_dtype)
    parts, f16, e4m3 = _PRODUCTS[prec][1], prec == 'f16', prec == 'fp8'
    xp = x if isinstance(x, PackedAct) else pack_operand(x, prec)
    n, _, h, w = xp.shape
    out_h = (h - 1) * 2 - 2 * padding[0] + kh + output_padding[0]
    out_w = (w - 1) * 2 - 2 * padding[1] + kw + output_padding[1]
    out_dtype = src_dtype if src_dtype != torch.float64 else torch.float32
    y = torch.empty([n, oc, out_h, out_w], dtype=out_dtype, device=xp.device)
    for ph in tconv_stride2_phase_plan(kh, kw, padding):
        view = y[:, :, ph['ry']::2, ph['rx']::2]
        if view.numel() == 0:
            continue
        if ph['ty'] == 0 or ph['tx'] == 0:          # no tap of the kernel reaches this phase (1-tap kernels)
            view.zero_()
            if bias is not None:
                view += bias.to(out_dtype).reshape(1, -1, 1, 1)
            continue
        def build(ph=ph):
            sub = weight.detach()[:, :, ph['t0y']::2, ph['t0x']::2].contiguous()
            return pack_weights_native(sub, ph['ty'], ph['tx'], parts, ph['pad_y'], ph['pad_x'], transpose_io=True, flip=True, scale=float(scale), f16=f16,
                                       e4m3=e4m3)
        pw = _cached(weight, ('tconv_phase', ph['ry'], ph['rx'], int(padding[0]), int(padding[1]), parts, f16, float(scale)) + (('e4m3',) if e4m3 else ()),
                     build)
        igemm_conv(xp, pw, out_hw=(int(view.shape[2]), int(view.shape[3])), out=view, bias=bias, precision=prec)
    if src_dtype == torch.float64:
        y = y.to(torch.float64)
    return y, xp


def _forward_conv_transpose(x, weight, bias, stride, padding, output_padding, keep=False, scale=1.0):
    """F.conv_transpose2d(x, weight[I, O, kh, kw], ...) as zero insertion + a stride-1 convolution with the
    flipped, transposed kernel (the data-gradient form; the fused up=2 layer does NOT come through here).
    x: tensor, or for stride 1 a PackedAct.  keep=True also returns the packed copy of x when the kernel consumed x itself
    (stride 1), else None."""
    from . import upfirdn2d as _up
    ic, oc, kh, kw = weight.shape
    sy, sx = stride
    if TCONV_PHASES and sy == 2 and sx == 2 and padding[0] <= kh - 1 and padding[1] <= kw - 1:
        y, xp = _conv_transpose_stride2_phases(x, weight, bias, padding, output_padding, scale)
        return (y, xp) if keep else y
    src_dtype = (torch.float16 if x.data.dtype == torch.float16 else weight.dtype) if isinstance(x, PackedAct) else x.dtype   # f16 operands: fp16 layer
    strided = sy > 1 or sx > 1
    if strided:
        assert not isinstance(x, PackedAct)
        # insert zeros between samples; crop the trailing (s-1) zeros the insertion appends
        x = _up.upfirdn2d(x, None, up=[sx, sy], padding=[0, -(sx - 1), 0, -(sy - 1)])
    py, px = kh - 1 - padding[0], kw - 1 - padding[1]
    assert py >= 0 and px >= 0, 'conv_transpose2d padding larger than kernel_size-1 is not supported'
    prec = precision_for(src_dtype)
    pw = packed_plain(weight, False, _PRODUCTS[prec][1], py, px, transpose_io=True, f16=prec == 'f16', scale=scale,    # flipped + transposed =
                      e4m3=prec == 'fp8')                                                                                # equivalent correlation kernel
    n, _, h, w = x.shape
    out_h = h + 2 * py - kh + 1 + output_padding[0]
    out_w = w + 2 * px - kw + 1 + output_padding[1]
    xp, mf = x, None
    if keep and not strided and not isinstance(x, PackedAct):
        mf = torch.channels_last if (x.stride(1) == 1 and x.shape[1] > 1) else torch.contiguous_format
        xp = pack_operand(x, prec)
    y = igemm_conv(xp, pw, stride=1, bias=bias, out_hw=(out_h, out_w), precision=prec, out_dtype=src_dtype if src_dtype != torch.float64 else None,
                   memory_format=mf)
    if src_dtype == torch.float64 and y.dtype != torch.float64:
        y = y.to(torch.float64)
    if keep:
        return y, (xp if isinstance(xp, PackedAct) else None)
    return y


def weight_gradient(grad_output, input, weight_shape, stride, padding, transpose, precision=None, out_dtype=None, dil_y=1, out_scale=1.0):
    """dW of conv2d (transpose=False, weight [O, I, kh, kw]) or conv_transpose2d (transpose=True, weight [I, O, kh, kw]):
    what Conv2dGradWeight.forward (conv2d_gradfix.py:135-142) gets from cuDNN, computed by pgpp_conv2d_wgrad as
    G[a, b, ky, kx] = sum S[n, a, y, x] * L[n, b, y*s + ky - p, x*s + kx - p] with (S, L) = (grad_output, input) for the
    convolution and (input, grad_output) for the transposed convolution."""
    _init()
    if out_dtype is None:
        out_dtype = next(t.dtype for t in (input, grad_output) if not isinstance(t, PackedAct))
    precision = precision or precision_for(out_dtype)
    products, parts = _PRODUCTS[precision]
    small, large = (input, grad_output) if transpose else (grad_output, input)
    ca, cb, kh, kw = (int(v) for v in weight_shape)
    n = int(small.shape[0])
    assert small.shape[1] == ca and large.shape[1] == cb and large.shape[0] == n
    ca_pad, cb_pad = _round_up(ca, 64), _round_up(cb, 64)
    f16 = precision == 'f16'
    s_op = small if isinstance(small, PackedAct) else pack_operand(small, precision)      # operands the forward / data-gradient kernels
    l_op = large if isinstance(large, PackedAct) else pack_operand(large, precision)      # already packed are used as they are
    for op, cpad in ((s_op, ca_pad), (l_op, cb_pad)):
        assert op.data.shape[0] >= parts and op.data.shape[4] - op.c_off >= cpad and (op.data.dtype == torch.float16) == f16
    device = s_op.data.device
    out = torch.empty([ca, cb, kh, kw], dtype=torch.float32, device=device)
    d = custom_ops.WgradDesc()
    d.small = s_op.data.data_ptr() + 2 * s_op.c_off; d.large = l_op.data.data_ptr() + 2 * l_op.c_off
    d.s_parts = s_op.data.shape[0]; d.l_parts = l_op.data.shape[0]
    d.n = n
    d.ca = ca; d.ca_pad = ca_pad; d.s_pixel_stride = s_op.data.shape[4]; d.hs = int(small.shape[2]); d.ws = int(small.shape[3])
    d.cb = cb; d.cb_pad = cb_pad; d.l_pixel_stride = l_op.data.shape[4]; d.hl = int(large.shape[2]); d.wl = int(large.shape[3])
    d.kh = kh; d.kw = kw; d.pad_y = int(padding[0]); d.pad_x = int(padding[1])
    d.stride = int(stride); d.products = products; d.operand_f16 = int(f16); d.dil_y = int(dil_y); d.out_scale = float(out_scale)
    workspace = torch.empty([kh * kw, ca, cb_pad], dtype=torch.float32, device=device)
    d.out = out.data_ptr(); d.workspace = workspace.data_ptr()
    if trace is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    _plugin.conv2d_wgrad(d, device)
    if trace is not None:
        e1.record()
        flops = 2.0 * n * small.shape[2] * small.shape[3] * ca * cb * kh * kw
        trace.append((f'wgrad {ca}x{cb} k{kh} {small.shape[2]}x{small.shape[3]} s{stride} n{n} {precision}', flops, e0, e1))
    return out if out_dtype == torch.float32 else out.to(out_dtype)


_conv2d_gradfix_cache = dict()


def _conv2d_gradfix(transpose, weight_shape, stride, padding, output_padding, dilation, groups, weight_scale=1.0, epilogue=None):
    ndim = 2
    weight_shape = tuple(weight_shape)
    stride = _tuple_of_ints(stride, ndim)
    padding = _tuple_of_ints(padding, ndim)
    output_padding = _tuple_of_ints(output_padding, ndim)
    dilation = _tuple_of_ints(dilation, ndim)
    key = (transpose, weight_shape, stride, padding, output_padding, dilation, groups, weight_scale, epilogue)
    if key in _conv2d_gradfix_cache:
        return _conv2d_gradfix_cache[key]

    assert groups >= 1
    assert len(weight_shape) == ndim + 2
    assert all(s >= 1 for s in stride)
    assert all(p >= 0 for p in padding)
    assert all(d >= 0 for d in dilation)
    if not transpose:
        assert all(p == 0 for p in output_padding)
    else:
        assert all(0 <= output_padding[i] < max(stride[i], dilation[i]) for i in range(ndim))
    if groups != 1 or any(d != 1 for d in dilation) or stride[0] != stride[1] or stride[0] > 2:
        raise NotImplementedError('the sm_100a convolution supports groups=1, dilation=1, stride 1 or 2; '
                                  'set conv2d_gradfix.enabled = False to route this call to the PyTorch library op')

    common_kwargs = dict(stride=stride, padding=padding, dilation=dilation, groups=groups, weight_scale=weight_scale)
    epi = epi_grad = None
    if epilogue is not None:
        assert not transpose
        from . import bias_act as _ba
        e_act, e_alpha, e_gain, e_clamp = epilogue
        epi = dict(act=e_act, alpha=e_alpha, gain=e_gain, clamp=e_clamp)
        _ba._init()
        fn = _ba._bias_act_cuda(dim=1, act=e_act, alpha=e_alpha, gain=e_gain, clamp=e_clamp if e_clamp >= 0 else None)
        epi_grad = None if fn.is_identity else fn.Grad      # d(pre-activation) = Grad(dy; y): linear in dy, differentiable once more
        epi_null, epi_keep_y = _ba._null_tensor, fn.keep_y

    def calc_output_padding(input_shape, output_shape):
        if transpose:
            return [0, 0]
        return [input_shape[i + 2] - (output_shape[i + 2] - 1) * stride[i] - (1 - 2 * padding[i])
                - dilation[i] * (weight_shape[i + 2] - 1) for i in range(ndim)]

    class Conv2d(torch.autograd.Function):
        @staticmethod
        def forward(ctx, input, weight, bias):
            assert weight.shape == weight_shape
            keep = keep_packed_operands and ctx.needs_input_grad[1]
            ctx.input_packed = None
            if not transpose:
                output = _forward_conv(input, weight, bias, stride, padding, keep=keep, scale=weight_scale, epi=epi)
            else:
                output = _forward_conv_transpose(input, weight, bias, stride, padding, output_padding, keep=keep, scale=weight_scale)
            if keep:
                output, ctx.input_packed = output
            if epi_grad is not None and epi_keep_y:
                ctx.save_for_backward(input, weight, output)
            else:
                ctx.save_for_backward(input, weight)
            return output

        @staticmethod
        def backward(ctx, grad_output):
            input, weight = ctx.saved_tensors[:2]
            grad_input = grad_weight = grad_bias = None
            want_w = ctx.needs_input_grad[1] and not weight_gradients_disabled
            plain = not torch.is_grad_enabled() and keep_packed_operands
            go_shape, go_dtype = grad_output.shape, grad_output.dtype
            # the packed copy of grad_output feeds the data-gradient kernel where that one reads the operand format, and the weight gradient
            go_feeds_dgrad = ctx.needs_input_grad[0] and (transpose or stride[0] == 1 or (TCONV_PHASES and stride[0] == 2))
            go = None
            if epi_grad is not None:        # through the fused bias_act first: everything below sees the gradient of the pre-activation
                y = ctx.saved_tensors[2] if epi_keep_y else epi_null
                if (plain and FUSE_ACT_GRAD_PACK and epi_keep_y and (want_w or go_feeds_dgrad) and (go_feeds_dgrad or not ctx.needs_input_grad[0])
                        and grad_output.dtype in (torch.float32, torch.float16, torch.bfloat16) and y.dtype == grad_output.dtype
                        and y.is_contiguous() and y.shape[1] > 1):
                    # plain backward pass: dy * act'(y) goes straight into the operand format (one pass over dy and y; the NCHW gradient of
                    # the pre-activation is never written), the bias gradient from the same pass
                    prec = precision_for(go_dtype)
                    data, sums = _plugin.pack_act_gradient(grad_output.contiguous(), y, _ACT_IDX[epi['act']], epi['alpha'], epi['gain'], epi['clamp'],
                                                           _round_up(go_shape[1], 64), _PRODUCTS[prec][1], f16=prec == 'f16',
                                                           want_sums=ctx.needs_input_grad[2])
                    go = PackedAct(data, go_shape[1])
                    if ctx.needs_input_grad[2]:
                        grad_bias = sums.sum([0, 2]).to(go_dtype)
                    grad_output = None
                else:
                    mf = torch.channels_last if (epi_keep_y and y.stride(1) == 1 and y.shape[1] > 1) else torch.contiguous_format
                    grad_output = epi_grad.apply(grad_output.contiguous(memory_format=mf), epi_null, epi_null, y)
            if plain:
                # plain backward pass (no graph is being recorded): grad_output is packed once and feeds both the data-gradient and
                # the weight-gradient kernel; the weight gradient reads the input operand the forward pass kept
                prec = precision_for(go_dtype)
                if go is None and (want_w or go_feeds_dgrad):
                    go = pack_operand(grad_output, prec)
                if ctx.needs_input_grad[0]:
                    p = calc_output_padding(input_shape=input.shape, output_shape=go_shape)
                    if transpose:       # gradient of conv_transpose2d = conv2d of grad_output with the same weight
                        grad_input = _forward_conv(go, weight, None, stride, padding, scale=weight_scale)
                    else:               # gradient of conv2d = conv_transpose2d (zero insertion first when strided)
                        grad_input = _forward_conv_transpose(go if go_feeds_dgrad else grad_output, weight, None,
                                                             stride, padding, p, scale=weight_scale)
                    assert grad_input.shape == input.shape
                if want_w:
                    xin = ctx.input_packed if ctx.input_packed is not None else input
                    if isinstance(xin, PackedAct) and xin.im2col is not None:
                        grad_weight = _weight_gradient_im2col(go, xin, weight_shape, xin.im2col, prec, weight.dtype)
                        if weight_scale != 1.0:
                            grad_weight = grad_weight * weight_scale
                    else:       # the runtime weight gain leaves with the gradient (pgpp_wgrad_desc.out_scale)
                        grad_weight = weight_gradient(go, xin, weight_shape, stride[0], padding, transpose, precision=prec, out_dtype=weight.dtype,
                                                      out_scale=weight_scale)
                    assert grad_weight.shape == weight_shape
                ctx.input_packed = None
            else:
                if ctx.needs_input_grad[0]:
                    p = calc_output_padding(input_shape=input.shape, output_shape=grad_output.shape)
                    grad_input = _conv2d_gradfix(transpose=(not transpose), weight_shape=weight_shape, output_padding=p,
                                                 **common_kwargs).apply(grad_output, weight, None)
                    assert grad_input.shape == input.shape
                if want_w:
                    grad_weight = Conv2dGradWeight.apply(grad_output, input)
                    if grad_weight.dtype != weight.dtype:
                        grad_weight = grad_weight.to(weight.dtype)
                    assert grad_weight.shape == weight_shape
            if ctx.needs_input_grad[2] and grad_bias is None:
                if (grad_output.is_contiguous() and grad_output.dtype in (torch.float32, torch.float16, torch.bfloat16) and
                        grad_output.shape[2] * grad_output.shape[3] >= 1024 and not (torch.is_grad_enabled() and grad_output.requires_grad)):
                    grad_bias = _plugin.sum_hw(grad_output).sum(0).to(grad_output.dtype)
                else:
                    grad_bias = grad_output.sum([0, 2, 3])
            return grad_input, grad_weight, grad_bias

    class Conv2dGradWeight(torch.autograd.Function):
        @staticmethod
        def forward(ctx, grad_output, input):
            gw = weight_gradient(grad_output, input, weight_shape, stride[0], padding, transpose, out_scale=weight_scale)
            assert gw.shape == weight_shape
            ctx.save_for_backward(grad_output, input)
            return gw

        @staticmethod
        def backward(ctx, grad2_grad_weight):
            grad_output, input = ctx.saved_tensors
            grad2_grad_output = grad2_input = None
            if ctx.needs_input_grad[0]:
                grad2_grad_output = Conv2d.apply(input, grad2_grad_weight, None)
                assert grad2_grad_output.shape == grad_output.shape
            if ctx.needs_input_grad[1]:
                p = calc_output_padding(input_shape=input.shape, output_shape=grad_output.shape)
                grad2_input = _conv2d_gradfix(transpose=(not transpose), weight_shape=weight_shape, output_padding=p,
                                              **common_kwargs).apply(grad_output, grad2_grad_weight, None)
                assert grad2_input.shape == input.shape
            return grad2_grad_output, grad2_input

    _conv2d_gradfix_cache[key] = Conv2d
    return Conv2d
