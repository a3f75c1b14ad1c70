"""Plugin loader: hands out the PREBUILT sm_100a C-ABI library instead of JIT-compiling sources.

Replaces the reference's torch_utils/custom_ops.py:46-124 (ninja JIT + importlib; broken on
torch 2.x).  `get_plugin(name)` keeps its name and caching behaviour but returns a thin object whose
methods have the signatures of the reference's pybind functions (bias_act.cpp:32, upfirdn2d.cpp:16)
and forward to `extern "C"` entry points of lib/libpgpp_sm100a.so (include/pgpp.h) through ctypes.
There is no fallback: if the library is missing or the call fails, a RuntimeError is raised.
"""
import ctypes
import os

import torch

verbosity = 'brief'     # 'none', 'brief', 'full' -- kept for compatibility (custom_ops.py:23)

# What `impl='cuda'` does with a NON-CUDA tensor.  'raise' (default): RuntimeError -- nothing is ever silently computed off the
# kernels.  'ref': the reference's own dispatch rule (bias_act.py:87, upfirdn2d.py:162: "cuda iff the tensor is on a CUDA device,
# else the ref path"), so that reference model code runs unchanged on CPU tensors through `pgpp_b200.install(cpu_tensors='ref')`.
# CUDA tensors are unaffected by this switch: they reach the sm_100a kernel or raise.
cpu_tensors = 'raise'

_LIB_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'lib', 'libpgpp_sm100a.so')
_lib = None
_cached_plugins = dict()

_DTYPES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2, torch.float64: 3, torch.float8_e4m3fn: 4}

c_i64x4 = ctypes.c_int64 * 4


class ConvDesc(ctypes.Structure):
    """mirror of pgpp_conv_desc (include/pgpp.h)"""
    _fields_ = [
        ('act', ctypes.c_void_p), ('wgt', ctypes.c_void_p),
        ('a_parts', ctypes.c_int32), ('b_parts', ctypes.c_int32),
        ('n', ctypes.c_int32), ('h', ctypes.c_int32), ('w', ctypes.c_int32), ('c_pad', ctypes.c_int32),
        ('act_pixel_stride', ctypes.c_int32), ('wgt_per_sample', ctypes.c_int32),
        ('kh', ctypes.c_int32), ('kw', ctypes.c_int32),
        ('pad_y', ctypes.c_int32), ('pad_x', ctypes.c_int32),
        ('stride', ctypes.c_int32), ('dil_y', ctypes.c_int32),
        ('conv_h', ctypes.c_int32), ('conv_w', ctypes.c_int32),
        ('o', ctypes.c_int32), ('phases', ctypes.c_int32), ('phase_stride', ctypes.c_int32), ('o_rows', ctypes.c_int32), ('block_n', ctypes.c_int32),
        ('products', ctypes.c_int32),
        ('dcoef', ctypes.c_void_p), ('noise', ctypes.c_void_p), ('noise_stride_n', ctypes.c_int64), ('bias', ctypes.c_void_p),
        ('act_fn', ctypes.c_int32), ('alpha', ctypes.c_float), ('gain', ctypes.c_float), ('clamp', ctypes.c_float),
        ('out', ctypes.c_void_p), ('out_dtype', ctypes.c_int32), ('out_h', ctypes.c_int32), ('out_w', ctypes.c_int32),
        ('out_stride', ctypes.c_int64 * 4),
        ('accumulate', ctypes.c_int32), ('out_parts', ctypes.c_int32), ('out_part_stride', ctypes.c_int64),
        ('spade_x', ctypes.c_void_p), ('spade_mean', ctypes.c_void_p), ('spade_rstd', ctypes.c_void_p), ('spade_pre_gain', ctypes.c_float),
        ('operand_f16', ctypes.c_int32),
        ('stats_ws', ctypes.c_void_p),
        ('wscale', ctypes.c_void_p), ('operand_e4m3', ctypes.c_int32), ('reserved1', ctypes.c_int32),
    ]


def library_path():
    return _LIB_PATH


def load_library():
    """dlopen the prebuilt library and declare the C prototypes.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(_LIB_PATH):
        raise RuntimeError(f'{_LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                           f'(or `make -C pasta-gan-plusplus_b200/csrc`). There is no fallback implementation.')
    lib = ctypes.CDLL(_LIB_PATH)
    vp, i64, i32, f32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_float
    lib.pgpp_version.restype = i32
    lib.pgpp_last_error.restype = ctypes.c_char_p
    lib.pgpp_launch_count.restype = i64
    lib.pgpp_refresh_env.restype = None
    lib.pgpp_bias_act.restype = i32
    lib.pgpp_bias_act.argtypes = [vp, vp, vp, vp, vp, vp, i64, i64, i64, i32, i32, i32, f32, f32, f32, vp]
    lib.pgpp_upfirdn2d.restype = i32
    lib.pgpp_upfirdn2d.argtypes = [vp, vp, vp, c_i64x4, c_i64x4, c_i64x4, c_i64x4, i32, i32, i64, i64,
                                   i32, i32, i32, i32, i32, i32, i32, f32, i32, vp]
    lib.pgpp_modconv_demod_coefs.restype = i32
    lib.pgpp_modconv_demod_coefs.argtypes = [vp, vp, vp, i32, i32, i32, i32, f32, vp]
    lib.pgpp_pack_activations.restype = i32
    lib.pgpp_pack_activations.argtypes = [vp, c_i64x4, c_i64x4, i32, vp, vp, i32, i32, vp]
    lib.pgpp_pack_activations_slice.restype = i32
    lib.pgpp_pack_activations_slice.argtypes = [vp, c_i64x4, c_i64x4, i32, vp, vp, i32, i32, i32, i32, vp]
    lib.pgpp_pack_activations_f16.restype = i32
    lib.pgpp_pack_activations_f16.argtypes = [vp, c_i64x4, c_i64x4, i32, vp, vp, i32, i32, i32, vp]
    lib.pgpp_pack_activations_e4m3.restype = i32
    lib.pgpp_pack_activations_e4m3.argtypes = [vp, c_i64x4, c_i64x4, i32, vp, vp, i32, i32, i32, vp]
    lib.pgpp_quantize_weights_e4m3.restype = i32
    lib.pgpp_quantize_weights_e4m3.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp]
    lib.pgpp_pack_weights.restype = i32
    lib.pgpp_pack_weights.argtypes = [vp, i32, c_i64x4, c_i64x4, i32, i32, f32, i32, i32, vp, i32, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.pgpp_up2_weight_adjoint.restype = i32
    lib.pgpp_up2_weight_adjoint.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp]
    lib.pgpp_pack_act_gradient.restype = i32
    lib.pgpp_pack_act_gradient.argtypes = [vp, vp, c_i64x4, c_i64x4, i32, i32, f32, f32, f32, vp, i32, i32, i32, vp, vp]
    lib.pgpp_pack_act_gradient_tiles.restype = i32
    lib.pgpp_pack_act_gradient_tiles.argtypes = [i32, i32]
    lib.pgpp_sum_hw.restype = i32
    lib.pgpp_sum_hw.argtypes = [vp, i32, vp, i32, i32, i64, vp]
    lib.pgpp_mul_reduce_hw.restype = i32
    lib.pgpp_mul_reduce_hw.argtypes = [vp, vp, vp, i64, vp, vp, vp, i32, i32, i64, vp]
    lib.pgpp_modulate_weights.restype = i32
    lib.pgpp_modulate_weights.argtypes = [vp, vp, vp, i32, i64, i32, i32, i32, vp]
    lib.pgpp_pack_im2col.restype = i32
    lib.pgpp_pack_im2col.argtypes = [vp, c_i64x4, c_i64x4, i32, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.pgpp_spade_modulate_pack.restype = i32
    lib.pgpp_spade_modulate_pack.argtypes = [vp, vp, vp, vp, vp, i64, vp, i32, i32, i32, i32, i32, i32, f32, vp]
    lib.pgpp_mix_pack.restype = i32
    lib.pgpp_mix_pack.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.pgpp_fir_pack.restype = i32
    lib.pgpp_fir_pack.argtypes = [vp, c_i64x4, c_i64x4, ctypes.POINTER(ctypes.c_float), i32, i32, i32, i32, i32, i32, i32, f32, vp, i32, i32, vp]
    lib.pgpp_fir_packed.restype = i32
    lib.pgpp_fir_packed.argtypes = [vp, i32, i64, i32, i32, i32, i32, i32, ctypes.POINTER(ctypes.c_float), i32, i32, i32, i32, i32, i32, i32, i32, f32,
                                    vp, i32, i64, i32, vp]
    lib.pgpp_fir_packed_act.restype = i32
    lib.pgpp_fir_packed_act.argtypes = [vp, i32, i64, i32, i32, i32, i32, i32, ctypes.POINTER(ctypes.c_float), i32, i32, i32, i32, i32, i32, i32, f32,
                                        vp, i64, vp, i32, f32, f32, f32, vp, i32, i64, i32, vp, i32, vp]
    lib.pgpp_conv1x1_thin.restype = i32
    lib.pgpp_conv1x1_thin.argtypes = [vp, i32, i64, i32, i32, i32, i64, vp, vp, i32, vp, i32, vp, vp, i32, vp, vp, i32, f32, f32, f32, vp]
    lib.pgpp_conv2d_direct.restype = i32
    lib.pgpp_conv2d_direct.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, f32, i32, f32, f32, f32, vp, vp, i32, i32, i32, vp]
    lib.pgpp_conv2d_igemm.restype = i32
    lib.pgpp_conv2d_igemm.argtypes = [ctypes.POINTER(ConvDesc), vp]
    lib.pgpp_conv2d_igemm_stats_rows.restype = i64
    lib.pgpp_conv2d_igemm_stats_rows.argtypes = [ctypes.POINTER(ConvDesc)]
    lib.pgpp_instnorm_finalize.restype = i32
    lib.pgpp_instnorm_finalize.argtypes = [vp, i64, i32, i32, f32, vp, vp, vp]
    lib.pgpp_conv2d_wgrad.restype = i32
    lib.pgpp_conv2d_wgrad.argtypes = [ctypes.POINTER(WgradDesc), vp]
    lib.pgpp_u8_to_f32.restype = i32
    lib.pgpp_u8_to_f32.argtypes = [vp, i64, i64, i64, vp, i64, i64, i32, vp, vp]
    lib.pgpp_image_to_u8.restype = i32
    lib.pgpp_image_to_u8.argtypes = [vp, i64, i64, i64, vp, i32, vp]
    lib.pgpp_grid_sample_2d.restype = i32
    lib.pgpp_grid_sample_2d.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.pgpp_grid_sample_2d_backward.restype = i32
    lib.pgpp_grid_sample_2d_backward.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]
    _lib = lib
    return lib


EXPORTED_SYMBOLS = ('pgpp_version', 'pgpp_last_error', 'pgpp_launch_count', 'pgpp_refresh_env', 'pgpp_bias_act', 'pgpp_upfirdn2d',
                    'pgpp_modconv_demod_coefs', 'pgpp_pack_activations', 'pgpp_pack_activations_slice', 'pgpp_pack_activations_f16', 'pgpp_pack_activations_e4m3', 'pgpp_quantize_weights_e4m3', 'pgpp_pack_act_gradient', 'pgpp_pack_act_gradient_tiles',
                    'pgpp_pack_weights', 'pgpp_up2_weight_adjoint', 'pgpp_mul_reduce_hw', 'pgpp_sum_hw', 'pgpp_modulate_weights',
                    'pgpp_spade_modulate_pack', 'pgpp_mix_pack', 'pgpp_conv2d_direct', 'pgpp_fir_pack', 'pgpp_fir_packed', 'pgpp_fir_packed_act', 'pgpp_conv1x1_thin', 'pgpp_pack_im2col', 'pgpp_conv2d_igemm', 'pgpp_conv2d_igemm_stats_rows', 'pgpp_instnorm_finalize', 'pgpp_conv2d_wgrad', 'pgpp_u8_to_f32',
                    'pgpp_image_to_u8', 'pgpp_grid_sample_2d', 'pgpp_grid_sample_2d_backward')


class WgradDesc(ctypes.Structure):
    """mirror of pgpp_wgrad_desc (include/pgpp.h)"""
    _fields_ = [
        ('small', ctypes.c_void_p), ('large', ctypes.c_void_p),
        ('s_parts', ctypes.c_int32), ('l_parts', ctypes.c_int32),
        ('n', ctypes.c_int32),
        ('ca', ctypes.c_int32), ('ca_pad', ctypes.c_int32), ('s_pixel_stride', ctypes.c_int32),
        ('hs', ctypes.c_int32), ('ws', ctypes.c_int32),
        ('cb', ctypes.c_int32), ('cb_pad', ctypes.c_int32), ('l_pixel_stride', ctypes.c_int32),
        ('hl', ctypes.c_int32), ('wl', ctypes.c_int32),
        ('kh', ctypes.c_int32), ('kw', ctypes.c_int32), ('pad_y', ctypes.c_int32), ('pad_x', ctypes.c_int32),
        ('stride', ctypes.c_int32), ('products', ctypes.c_int32),
        ('out', ctypes.c_void_p), ('workspace', ctypes.c_void_p),
        ('operand_f16', ctypes.c_int32), ('dil_y', ctypes.c_int32),
        ('out_scale', ctypes.c_float), ('reserved0', ctypes.c_int32),
    ]


def launch_count():
    return int(load_library().pgpp_launch_count())


def refresh_env():
    """re-read the PGPP_* ablation switches from os.environ (the library caches them at load time)"""
    load_library().pgpp_refresh_env()


def _check(status):
    if status != 0:
        raise RuntimeError(load_library().pgpp_last_error().decode())


def _torch_check(cond, msg):
    if not cond:
        raise RuntimeError(msg)


def _stream(t):
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None and t.numel() > 0 else None


def _same_layout(a, b):
    if a.dim() != b.dim():
        return False
    return all(sa == sb and (sa < 2 or ta == tb) for sa, sb, ta, tb in zip(a.shape, b.shape, a.stride(), b.stride()))


def _is_dense(t):
    """non-overlapping and dense (any dimension order), like at::Tensor::is_non_overlapping_and_dense"""
    dims = sorted(((st, sz) for sz, st in zip(t.shape, t.stride()) if sz > 1))
    expect = 1
    for st, sz in dims:
        if st != expect:
            return False
        expect *= sz
    return True


def dtype_code(dtype):
    _torch_check(dtype in _DTYPES, f'unsupported dtype {dtype}')
    return _DTYPES[dtype]


class _BiasActPlugin:
    """`bias_act(x, b, xref, yref, dy, grad, dim, act, alpha, gain, clamp) -> Tensor`; validation follows
    torch_utils/ops/bias_act.cpp:35-51, empty tensors mean "absent" (bias_act.py:39)."""

    @staticmethod
    def bias_act(x, b, xref, yref, dy, grad, dim, act, alpha, gain, clamp):
        lib = load_library()
        _torch_check(x.is_cuda, 'x must reside on CUDA device')
        _torch_check(b.numel() == 0 or (b.dtype == x.dtype and b.device == x.device), 'b must have the same dtype and device as x')
        for t, name in ((xref, 'xref'), (yref, 'yref'), (dy, 'dy')):
            _torch_check(t.numel() == 0 or (t.shape == x.shape and t.dtype == x.dtype and t.device == x.device),
                         f'{name} must have the same shape, dtype, and device as x')
        _torch_check(x.numel() <= 2 ** 31 - 1, 'x is too large')
        _torch_check(b.dim() == 1, 'b must have rank 1')
        _torch_check(b.numel() == 0 or (0 <= dim < x.dim()), 'dim is out of bounds')
        _torch_check(b.numel() == 0 or b.numel() == x.shape[dim], 'b has wrong number of elements')
        _torch_check(grad >= 0, 'grad must be non-negative')
        _torch_check(_is_dense(x), 'x must be non-overlapping and dense')
        _torch_check(b.is_contiguous(), 'b must be contiguous')
        for t, name in ((xref, 'xref'), (yref, 'yref'), (dy, 'dy')):
            _torch_check(t.numel() == 0 or _same_layout(t, x), f'{name} must have the same layout as x')
        y = torch.empty_like(x)
        _torch_check(_same_layout(y, x), 'y must have the same layout as x')
        step_b = x.stride(dim) if b.numel() else 1
        with torch.cuda.device(x.device):
            _check(lib.pgpp_bias_act(_ptr(x), _ptr(b), _ptr(xref), _ptr(yref), _ptr(dy), _ptr(y), x.numel(), b.numel(),
                                     step_b, dtype_code(x.dtype), int(grad), int(act), float(alpha), float(gain),
                                     float(clamp), _stream(x)))
        return y


class _Upfirdn2dPlugin:
    """`upfirdn2d(x, f, upx, upy, downx, downy, padx0, padx1, pady0, pady1, flip, gain) -> Tensor`; validation
    and output size follow torch_utils/ops/upfirdn2d.cpp:19-36."""

    @staticmethod
    def upfirdn2d(x, f, upx, upy, downx, downy, padx0, padx1, pady0, pady1, flip, gain, row_align=1):
        """`row_align` > 1 (not in the reference): rows of the (NCHW) result start at multiples of `row_align` elements - the
        returned tensor is a [..., :out_w] view of a wider allocation - so that odd-width blur outputs (513 = 512 + 1 before
        a strided conv) keep 16-byte aligned rows for the kernels that follow."""
        lib = load_library()
        _torch_check(x.is_cuda, 'x must reside on CUDA device')
        _torch_check(f.device == x.device, 'f must reside on the same device as x')
        _torch_check(f.dtype == torch.float32, 'f must be float32')
        _torch_check(x.numel() <= 2 ** 31 - 1, 'x is too large')
        _torch_check(x.dim() == 4, 'x must be rank 4')
        _torch_check(f.dim() == 2, 'f must be rank 2')
        _torch_check(f.shape[0] >= 1 and f.shape[1] >= 1, 'f must be at least 1x1')
        _torch_check(upx >= 1 and upy >= 1, 'upsampling factor must be at least 1')
        _torch_check(downx >= 1 and downy >= 1, 'downsampling factor must be at least 1')
        n, c, h, w = x.shape
        out_w = (w * upx + padx0 + padx1 - f.shape[1] + downx) // downx
        out_h = (h * upy + pady0 + pady1 - f.shape[0] + downy) // downy
        _torch_check(out_w >= 1 and out_h >= 1, 'output must be at least 1x1')
        mf = torch.channels_last if (x.stride(1) == 1 and c > 1) else torch.contiguous_format
        if row_align > 1 and mf == torch.contiguous_format and out_w % row_align:
            y = torch.empty([n, c, out_h, -(-out_w // row_align) * row_align], dtype=x.dtype, device=x.device)[..., :out_w]
        else:
            y = torch.empty([n, c, out_h, out_w], dtype=x.dtype, device=x.device, memory_format=mf)
        _torch_check(y.numel() <= 2 ** 31 - 1, 'output is too large')
        with torch.cuda.device(x.device):
            _check(lib.pgpp_upfirdn2d(_ptr(x), _ptr(f), _ptr(y), c_i64x4(*x.shape), c_i64x4(*x.stride()),
                                      c_i64x4(*y.shape), c_i64x4(*y.stride()), f.shape[1], f.shape[0],
                                      f.stride(1), f.stride(0), int(upx), int(upy), int(downx), int(downy),
                                      int(padx0), int(pady0), int(bool(flip)), float(gain), dtype_code(x.dtype), _stream(x)))
        return y


class _ConvPlugin:
    """New entry points with no reference counterpart (they replace cuDNN calls, conv2d_gradfix.py:112-114)."""

    @staticmethod
    def demod_coefs(weight, styles, eps=1e-8):
        lib = load_library()
        o, i = weight.shape[0], weight.shape[1]
        w = weight.detach().to(torch.float32).contiguous()
        s = styles.detach().to(torch.float32).contiguous()
        d = torch.empty([s.shape[0], o], dtype=torch.float32, device=w.device)
        with torch.cuda.device(w.device):
            _check(lib.pgpp_modconv_demod_coefs(_ptr(w), _ptr(s), _ptr(d), s.shape[0], o, i, w[0, 0].numel(), float(eps), _stream(w)))
        return d

    @staticmethod
    def pack_activations(x, scale, c_pad, parts, f16=False, e4m3=False):
        """-> [parts, N, H, W, c_pad] bfloat16 parts; with f16=True one part of IEEE half (dtype float16); with e4m3=True one part of
        e4m3 bytes (dtype float8_e4m3fn, round to nearest even, |v| > 448 saturates)"""
        lib = load_library()
        _torch_check(x.is_cuda and x.dim() == 4, 'x must be a rank-4 CUDA tensor')
        n, c, h, w = x.shape
        if scale is not None:
            scale = scale.detach().to(torch.float32).contiguous()
            _torch_check(tuple(scale.shape) == (n, c), 'scale must be [N, C]')
        if e4m3:
            out = torch.empty([1, n, h, w, c_pad], dtype=torch.float8_e4m3fn, device=x.device)
            with torch.cuda.device(x.device):
                _check(lib.pgpp_pack_activations_e4m3(_ptr(x), c_i64x4(*x.shape), c_i64x4(*x.stride()), dtype_code(x.dtype),
                                                      _ptr(scale), _ptr(out), int(c_pad), int(c_pad), 0, _stream(x)))
            return out
        if f16:
            out = torch.empty([1, n, h, w, c_pad], dtype=torch.float16, device=x.device)
            with torch.cuda.device(x.device):
                _check(lib.pgpp_pack_activations_f16(_ptr(x), c_i64x4(*x.shape), c_i64x4(*x.stride()), dtype_code(x.dtype),
                                                     _ptr(scale), _ptr(out), int(c_pad), int(c_pad), 0, _stream(x)))
            return out
        out = torch.empty([parts, n, h, w, c_pad], dtype=torch.bfloat16, device=x.device)
        with torch.cuda.device(x.device):
            _check(lib.pgpp_pack_activations(_ptr(x), c_i64x4(*x.shape), c_i64x4(*x.stride()), dtype_code(x.dtype),
                                             _ptr(scale), _ptr(out), int(c_pad), int(parts), _stream(x)))
        return out

    @staticmethod
    def pack_act_gradient(dy, y, act_idx, alpha, gain, clamp, c_pad, parts, f16=False, want_sums=False):
        """operand-format copy of the gradient of a fused bias_act, from dy and the saved output y (see pgpp_pack_act_gradient);
        -> (packed [parts, N, H, W, c_pad], per-tile channel sums float32 [N, C, tiles] or None)"""
        lib = load_library()
        _torch_check(dy.is_cuda and dy.dim() == 4 and dy.shape == y.shape and dy.dtype == y.dtype and dy.stride() == y.stride(),
                     'dy and y must be rank-4 CUDA tensors of the same shape, dtype and strides')
        n, c, h, w = dy.shape
        out = torch.empty([1 if f16 else parts, n, h, w, c_pad], dtype=torch.float16 if f16 else torch.bfloat16, device=dy.device)
        sums = torch.empty([n, c, lib.pgpp_pack_act_gradient_tiles(h, w)], dtype=torch.float32, device=dy.device) if want_sums else None
        with torch.cuda.device(dy.device):
            _check(lib.pgpp_pack_act_gradient(_ptr(dy), _ptr(y), c_i64x4(*dy.shape), c_i64x4(*dy.stride()), dtype_code(dy.dtype), int(act_idx),
                                              float(alpha), float(gain), float(clamp), _ptr(out), int(c_pad), 1 if f16 else int(parts), int(bool(f16)),
                                              _ptr(sums), _stream(dy)))
        return out, sums

    @staticmethod
    def pack_weights(weight, out, master, *, transpose_io=False, flip=False, scale=1.0, phases=1, phase_stride=0, fir=None, flip_filter=False,
                     parts=1, f16=False, o_off=0):
        """weight [O, I, kh, kw] (or [I, O, kh, kw] with transpose_io) -> rows [o_off, ...) of out [parts, taps, o_rows, c_pad]
        (bfloat16 parts or one float16 part) and optionally master float32 [taps, o_rows, c_pad]; see pgpp_pack_weights"""
        lib = load_library()
        _torch_check(weight.is_cuda and weight.dim() == 4, 'weight must be a rank-4 CUDA tensor')
        if out is None:     # master only (the e4m3 route quantizes it with quantize_weights_e4m3)
            _torch_check(master is not None and master.dim() == 3, 'master [taps, o_rows, c_pad] is required when out is None')
            o_rows, c_pad = int(master.shape[1]), int(master.shape[2])
        else:
            _torch_check(out.dim() == 4 and out.is_contiguous() and out.dtype in (torch.bfloat16, torch.float16) and out.shape[0] >= parts,
                         'out must be a contiguous [parts, taps, o_rows, c_pad] 16-bit tensor')
            _torch_check((out.dtype == torch.float16) == bool(f16), 'fp16 operands need a float16 destination (and only then)')
            o_rows, c_pad = int(out.shape[2]), int(out.shape[3])
        w = weight.detach()
        if fir is not None:
            _torch_check(fir.is_cuda and fir.dtype == torch.float32 and tuple(fir.shape) == (4, 4), 'fir must be a float32 CUDA tensor [4, 4]')
            fir = fir.contiguous()
        _torch_check(master is None or (master.dtype == torch.float32 and master.is_contiguous() and (out is None or master.numel() == out[0].numel())),
                     'master must be a contiguous float32 tensor with taps * o_rows * c_pad elements')
        with torch.cuda.device(w.device):
            _check(lib.pgpp_pack_weights(_ptr(w), dtype_code(w.dtype), c_i64x4(*w.shape), c_i64x4(*w.stride()), int(bool(transpose_io)),
                                         int(bool(flip)), float(scale), int(phases), int(phase_stride), _ptr(fir), int(bool(flip_filter)),
                                         _ptr(out), _ptr(master), int(parts), int(bool(f16)), o_rows, int(o_off), c_pad,
                                         _stream(w)))
        return out

    @staticmethod
    def quantize_weights_e4m3(master, styles=None):
        """master float32 [taps, o_rows, c_pad], styles [N, c_in] or None -> (e4m3 bytes float8_e4m3fn [N, 1, taps, o_rows, c_pad] (N = 1 for
        shared weights), column scales float32 [N, o_rows]); see pgpp_quantize_weights_e4m3"""
        lib = load_library()
        _torch_check(master.dtype == torch.float32 and master.is_contiguous() and master.dim() == 3, 'master must be contiguous float32 [taps, o_rows, c_pad]')
        taps, o_rows, c_pad = (int(v) for v in master.shape)
        s = None if styles is None else styles.detach().to(torch.float32).contiguous()
        n, c_in = (1, c_pad) if s is None else (int(s.shape[0]), int(s.shape[1]))
        out = torch.empty([n, 1, taps, o_rows, c_pad], dtype=torch.float8_e4m3fn, device=master.device)
        scale = torch.empty([n, o_rows], dtype=torch.float32, device=master.device)
        with torch.cuda.device(master.device):
            _check(lib.pgpp_quantize_weights_e4m3(_ptr(master), _ptr(s), n, taps, o_rows, c_pad, c_in, _ptr(out), _ptr(scale), _stream(master)))
        return out, scale

    @staticmethod
    def sum_hw(a):
        """a [N, C, H, W] contiguous float32 / float16 / bfloat16 -> float32 [N, C] plane sums; see pgpp_sum_hw"""
        lib = load_library()
        n, c, h, w = a.shape
        r = torch.empty([n, c], dtype=torch.float32, device=a.device)
        with torch.cuda.device(a.device):
            _check(lib.pgpp_sum_hw(_ptr(a), dtype_code(a.dtype), _ptr(r), n, c, h * w, _stream(a)))
        return r

    @staticmethod
    def mul_reduce_hw(a, b=None, sub=None, scale=None, out_scaled=False, reduce=True):
        """a, b float32 [N,C,H,W] contiguous; sub [H,W] or [N,1,H,W]; scale [N,C] ->
        (r [N,C] = sum_hw a * (b - sub) or None, a * scale[n,c] or None); see pgpp_mul_reduce_hw"""
        lib = load_library()
        _torch_check(a.is_cuda and a.dtype == torch.float32 and a.dim() == 4, 'mul_reduce_hw: a must be a float32 CUDA tensor [N,C,H,W]')
        a = a.contiguous()
        n, c, h, w = a.shape
        if b is not None:
            _torch_check(b.dtype == torch.float32 and tuple(b.shape) == tuple(a.shape), 'mul_reduce_hw: b must match a')
            b = b.contiguous()
        sub_stride = 0
        if sub is not None:
            sub = sub.detach().to(torch.float32).contiguous()
            _torch_check(sub.numel() in (h * w, n * h * w), 'mul_reduce_hw: sub must be [H,W] or [N,1,H,W]')
            sub_stride = h * w if sub.numel() == n * h * w and n > 1 else 0
        if scale is not None:
            scale = scale.detach().to(torch.float32).contiguous()
            _torch_check(scale.numel() == n * c, 'mul_reduce_hw: scale must be [N,C]')
        r = torch.empty([n, c], dtype=torch.float32, device=a.device) if reduce else None
        out = torch.empty_like(a) if out_scaled else None
        if a.numel() == 0:
            return (r.zero_() if r is not None else None), out
        with torch.cuda.device(a.device):
            _check(lib.pgpp_mul_reduce_hw(_ptr(a), _ptr(b), _ptr(sub), int(sub_stride), _ptr(scale), _ptr(out), _ptr(r), n, c, h * w, _stream(a)))
        return r, out

    @staticmethod
    def up2_weight_adjoint(grad_polyphase, fir, flip_filter, flip, o, ic):
        """grad_polyphase float32 [4, O, I, 3, 3] -> grad_weight float32 [O, I, 3, 3]; see pgpp_up2_weight_adjoint"""
        lib = load_library()
        g = grad_polyphase.contiguous()
        _torch_check(g.dtype == torch.float32 and g.numel() == 36 * o * ic, 'grad_polyphase must be float32 [4, O, I, 3, 3]')
        out = torch.empty([o, ic, 3, 3], dtype=torch.float32, device=g.device)
        with torch.cuda.device(g.device):
            _check(lib.pgpp_up2_weight_adjoint(_ptr(g), _ptr(fir.contiguous()), int(bool(flip_filter)), int(bool(flip)), int(o), int(ic),
                                               _ptr(out), _stream(g)))
        return out

    @staticmethod
    def pack_activations_into(x, scale, dst, c_pad, c_off):
        """pack x (optionally * scale[n,c]) into channels [c_off, c_off + c_pad) of dst [parts, N, H, W, c_total]"""
        lib = load_library()
        n, c, h, w = x.shape
        parts, c_total = dst.shape[0], dst.shape[4]
        _torch_check(tuple(dst.shape[1:4]) == (n, h, w) and dst.dtype in (torch.bfloat16, torch.float8_e4m3fn) and dst.is_contiguous(),
                     'bad packed destination')
        if scale is not None:
            scale = scale.detach().to(torch.float32).contiguous()
        if dst.dtype == torch.float8_e4m3fn:        # one part of e4m3 bytes
            _torch_check(parts == 1, 'e4m3 operands are one part')
            with torch.cuda.device(x.device):
                _check(lib.pgpp_pack_activations_e4m3(_ptr(x), c_i64x4(*x.shape), c_i64x4(*x.stride()), dtype_code(x.dtype), _ptr(scale),
                                                      _ptr(dst), int(c_pad), int(c_total), int(c_off), _stream(x)))
            return dst
        with torch.cuda.device(x.device):
            _check(lib.pgpp_pack_activations_slice(_ptr(x), c_i64x4(*x.shape), c_i64x4(*x.stride()), dtype_code(x.dtype), _ptr(scale),
                                                   _ptr(dst), int(c_pad), int(c_total), int(c_off), int(parts), _stream(x)))
        return dst

    @staticmethod
    def pack_im2col(x, scale, kw, r, pad_x, pad_y, parts):
        """row-group im2col operand [parts, N, H + pad_y, W, 64] (see pgpp_pack_im2col)"""
        lib = load_library()
        n, c, h, w = x.shape
        _torch_check(r * kw * c <= 64, 'im2col packing needs r*kw*C <= 64')
        out = torch.empty([parts, n, h + pad_y, w, 64], dtype=torch.bfloat16, device=x.device)
        if scale is not None:
            scale = scale.detach().to(torch.float32).contiguous()
        with torch.cuda.device(x.device):
            _check(lib.pgpp_pack_im2col(_ptr(x), c_i64x4(*x.shape), c_i64x4(*x.stride()), dtype_code(x.dtype), _ptr(scale), _ptr(out),
                                        int(kw), int(r), int(pad_x), int(pad_y), int(parts), _stream(x)))
        return out

    @staticmethod
    def modulate_weights(master, styles, parts):
        """master float32 [rows, c_pad], styles [N, c_in] -> bf16 [N, parts, rows, c_pad]"""
        lib = load_library()
        rows, c_pad = master.shape
        s = styles.detach().to(torch.float32).contiguous()
        out = torch.empty([s.shape[0], parts, rows, c_pad], dtype=torch.bfloat16, device=master.device)
        with torch.cuda.device(master.device):
            _check(lib.pgpp_modulate_weights(_ptr(master), _ptr(s), _ptr(out), s.shape[0], rows, c_pad, s.shape[1], int(parts), _stream(master)))
        return out

    @staticmethod
    def spade_modulate_pack(x, mean, rstd, gamma_beta, c_pad, parts, pre_gain):
        """x [N,C,H,W] f32 contiguous, gamma_beta [N,2C,H,W] f32 contiguous (gamma | beta), mean / rstd [N,C] ->
        bf16 [parts, N, H, W, c_pad] = split(pre_act((x-mean)*rstd*(1+gamma)+beta))"""
        lib = load_library()
        n, c, h, w = x.shape
        _torch_check(x.dtype == torch.float32 and x.is_contiguous() and gamma_beta.is_contiguous() and
                     tuple(gamma_beta.shape) == (n, 2 * c, h, w), 'spade_modulate_pack: bad operands')
        mean = mean.to(torch.float32).contiguous(); rstd = rstd.to(torch.float32).contiguous()
        if c_pad == c:
            out = torch.empty([parts, n, h, w, c_pad], dtype=torch.bfloat16, device=x.device)
        else:
            out = torch.zeros([parts, n, h, w, c_pad], dtype=torch.bfloat16, device=x.device)
        gamma_ptr = gamma_beta.data_ptr()
        beta_ptr = gamma_ptr + 4 * c * h * w
        with torch.cuda.device(x.device):
            _check(lib.pgpp_spade_modulate_pack(_ptr(x), _ptr(mean), _ptr(rstd), ctypes.c_void_p(gamma_ptr), ctypes.c_void_p(beta_ptr),
                                                2 * c * h * w, _ptr(out), n, c, h, w, int(c_pad), int(parts), float(pre_gain), _stream(x)))
        return out

    @staticmethod
    def conv2d_direct(x, weight, bias, wscale, act_idx, alpha, gain, clamp, out_packed_data=None, c_off=0):
        """exact-fp32 direct convolution for C*kh*kw <= 16 ('same' padding): returns float32 [N,O,H,W], or writes channels
        [c_off, c_off+O) of the operand-format buffer `out_packed_data` [parts,N,H,W,c_total]; see pgpp_conv2d_direct"""
        lib = load_library()
        _torch_check(x.is_cuda and x.dtype == torch.float32 and x.dim() == 4, 'conv2d_direct: x must be a float32 CUDA tensor [N,C,H,W]')
        x = x.contiguous()
        w = weight.detach().to(torch.float32).contiguous()
        n, c, h, wd = x.shape
        o, ic, kh, kw = w.shape
        _torch_check(ic == c, 'conv2d_direct: channel mismatch')
        b = bias.detach().to(torch.float32).contiguous() if bias is not None else None
        out = None
        if out_packed_data is None:
            out = torch.empty([n, o, h, wd], dtype=torch.float32, device=x.device)
            parts, c_total = 0, 0
        else:
            _torch_check(out_packed_data.dtype == torch.bfloat16 and tuple(out_packed_data.shape[1:4]) == (n, h, wd), 'conv2d_direct: bad packed destination')
            parts, c_total = out_packed_data.shape[0], out_packed_data.shape[4]
        with torch.cuda.device(x.device):
            _check(lib.pgpp_conv2d_direct(_ptr(x), _ptr(w), _ptr(b), n, c, h, wd, o, kh, kw, kh // 2, kw // 2, float(wscale), int(act_idx),
                                          float(alpha), float(gain), float(clamp), _ptr(out), _ptr(out_packed_data), int(c_total), int(c_off),
                                          int(parts), _stream(x)))
        return out

    @staticmethod
    def fir_pack(x, taps, fw, fh, padx0, padx1, pady0, pady1, flip, gain, c_pad, parts):
        """FIR blur (up = down = 1, `taps` = host list of fh * fw filter values) of x float32 [N,C,H,W] written as the operand
        format bf16 [parts, N, H', W', c_pad]; see pgpp_fir_pack"""
        lib = load_library()
        _torch_check(x.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and x.stride(3) == 1, 'fir_pack: x must be float32 [N,C,H,W] with unit W stride')
        n, c, h, w = x.shape
        oh, ow = h + pady0 + pady1 - fh + 1, w + padx0 + padx1 - fw + 1
        _torch_check(oh >= 1 and ow >= 1 and len(taps) == fw * fh, 'fir_pack: bad filter / padding')
        out = torch.empty([parts, n, oh, ow, c_pad], dtype=torch.bfloat16, device=x.device)
        f = (ctypes.c_float * (fw * fh))(*[float(t) for t in taps])
        with torch.cuda.device(x.device):
            _check(lib.pgpp_fir_pack(_ptr(x), c_i64x4(*x.shape), c_i64x4(*x.stride()), f, fw, fh, int(padx0), int(padx1), int(pady0), int(pady1),
                                     int(bool(flip)), float(gain), _ptr(out), int(c_pad), int(parts), _stream(x)))
        return out

    @staticmethod
    def conv1x1_thin(src, c, c_off, w1, b1, out1, accumulate1, w2=None, b2=None, out2=None, styles=None, act_idx=1, alpha=0.0, gain=1.0, clamp=-1.0):
        """1x1 modulated convolution with few output channels on the operand format (`src` bf16 [parts, N, H, W, c_total], channels
        [c_off, c_off + c)): out1 [N, o1, H, W] float32 (+= when accumulate1), optional second head out2 from w2 / b2; see pgpp_conv1x1_thin"""
        lib = load_library()
        _torch_check(src.is_cuda and src.dtype == torch.bfloat16 and src.dim() == 5 and src.is_contiguous(), 'conv1x1_thin: src must be a contiguous bf16 [parts,N,H,W,C] tensor')
        parts, n, h, w, ct = src.shape
        f32 = lambda t: None if t is None else t.detach().to(torch.float32).contiguous()
        w1, b1, w2, b2, styles = f32(w1), f32(b1), f32(w2), f32(b2), f32(styles)
        o1, o2 = int(w1.shape[0]), 0 if w2 is None else int(w2.shape[0])
        _torch_check(out1.dtype == torch.float32 and out1.is_contiguous() and tuple(out1.shape) == (n, o1, h, w), 'conv1x1_thin: out1 must be contiguous float32 [N,o1,H,W]')
        _torch_check(w1.numel() == o1 * c and (styles is None or tuple(styles.shape) == (n, c)), 'conv1x1_thin: weight / styles shape')
        if o2:
            _torch_check(out2 is not None and out2.dtype == torch.float32 and out2.is_contiguous() and tuple(out2.shape) == (n, o2, h, w) and w2.numel() == o2 * c,
                         'conv1x1_thin: out2 must be contiguous float32 [N,o2,H,W]')
        with torch.cuda.device(src.device):
            _check(lib.pgpp_conv1x1_thin(src.data_ptr() + 2 * c_off, int(parts), int(src[0].numel()), int(ct), n, int(c), h * w,
                                         _ptr(w1), _ptr(b1), o1, _ptr(out1), int(bool(accumulate1)), _ptr(w2), _ptr(b2), o2, _ptr(out2),
                                         _ptr(styles), int(act_idx), float(alpha), float(gain), float(clamp), _stream(src)))
        return out1, out2

    @staticmethod
    def fir_packed(src, c, c_off, taps, fw, fh, down, padx0, padx1, pady0, pady1, flip, gain, dst=None, dst_c_off=0, parts=None):
        """upfirdn2d (up = 1, down 1 or 2, filter at most 4 x 4 given as a host list, None = identity) on the operand format: channels
        [c_off, c_off + c) of `src` (bf16 [parts, N, H, W, c_total]) -> channels [dst_c_off, dst_c_off + c) of `dst` (allocated with
        c rounded up to whole 64-channel rows when None); see pgpp_fir_packed"""
        lib = load_library()
        _torch_check(src.is_cuda and src.dtype == torch.bfloat16 and src.dim() == 5 and src.is_contiguous(), 'fir_packed: src must be a contiguous bf16 [parts,N,H,W,C] tensor')
        sp, n, h, w, ct = src.shape
        oh, ow = (h + pady0 + pady1 - fh) // down + 1, (w + padx0 + padx1 - fw) // down + 1
        _torch_check(oh >= 1 and ow >= 1 and (taps is None or len(taps) == fw * fh), 'fir_packed: bad filter / padding')
        if dst is None:
            c_alloc = -(-c // 64) * 64
            alloc = torch.empty if c_alloc == c else torch.zeros
            dst = alloc([parts or sp, n, oh, ow, c_alloc], dtype=torch.bfloat16, device=src.device)
        _torch_check(dst.dtype == torch.bfloat16 and dst.is_contiguous() and tuple(dst.shape[1:4]) == (n, oh, ow), 'fir_packed: dst has the wrong shape')
        f = None if taps is None else (ctypes.c_float * (fw * fh))(*[float(t) for t in taps])
        with torch.cuda.device(src.device):
            _check(lib.pgpp_fir_packed(src.data_ptr() + 2 * c_off, int(sp), int(src[0].numel()), n, h, w, int(c), int(ct), f, int(fw), int(fh), int(down),
                                       int(padx0), int(padx1), int(pady0), int(pady1), int(bool(flip)), float(gain),
                                       dst.data_ptr() + 2 * dst_c_off, int(dst.shape[0]), int(dst[0].numel()), int(dst.shape[4]), _stream(src)))
        return dst

    @staticmethod
    def fir_packed_act(src, c, c_off, taps, fw, fh, padx0, padx1, pady0, pady1, flip, gain, noise, bias, act_idx, alpha, act_gain, clamp, dst, dst_c_off=0,
                       dst_nchw=None):
        """fir_packed (down = 1, separable filter) followed by clamp(act(v + noise + bias) * act_gain), written into channels
        [dst_c_off, dst_c_off + c) of `dst`; noise float32 [oh, ow] or [N, oh, ow] or None, bias float32 [c] or None; see pgpp_fir_packed_act"""
        lib = load_library()
        _torch_check(src.is_cuda and src.dtype == torch.bfloat16 and src.dim() == 5 and src.is_contiguous(), 'fir_packed_act: src must be a contiguous bf16 [parts,N,H,W,C] tensor')
        sp, n, h, w, ct = src.shape
        oh, ow = h + pady0 + pady1 - fh + 1, w + padx0 + padx1 - fw + 1
        if dst_nchw is not None:
            _torch_check(dst is None and dst_nchw.dtype == torch.float32 and dst_nchw.is_contiguous() and tuple(dst_nchw.shape) == (n, c, oh, ow),
                         'fir_packed_act: dst_nchw must be a contiguous float32 [N, c, oh, ow] tensor')
        else:
            _torch_check(dst.dtype == torch.bfloat16 and dst.is_contiguous() and tuple(dst.shape[1:4]) == (n, oh, ow), 'fir_packed_act: dst has the wrong shape')
        nz_stride = 0
        if noise is not None:
            noise = noise.detach().to(torch.float32).contiguous()
            _torch_check(noise.numel() in (oh * ow, n * oh * ow), 'fir_packed_act: noise must be [oh, ow] or [N, oh, ow]')
            nz_stride = oh * ow if (noise.numel() == n * oh * ow and n > 1) else 0
        if bias is not None:
            bias = bias.detach().to(torch.float32).contiguous()
            _torch_check(bias.numel() == c, 'fir_packed_act: bias must have c elements')
        f = (ctypes.c_float * (fw * fh))(*[float(t) for t in taps])
        with torch.cuda.device(src.device):
            _check(lib.pgpp_fir_packed_act(src.data_ptr() + 2 * c_off, int(sp), int(src[0].numel()), n, h, w, int(c), int(ct), f, int(fw), int(fh),
                                           int(padx0), int(padx1), int(pady0), int(pady1), int(bool(flip)), float(gain),
                                           _ptr(noise), int(nz_stride), _ptr(bias), int(act_idx), float(alpha), float(act_gain), float(clamp),
                                           None if dst is None else dst.data_ptr() + 2 * dst_c_off, 0 if dst is None else int(dst.shape[0]),
                                           0 if dst is None else int(dst[0].numel()), 0 if dst is None else int(dst.shape[4]),
                                           _ptr(dst_nchw), int(c), _stream(src)))
        return dst if dst is not None else dst_nchw

    @staticmethod
    def mix_pack(terms, c_pad, parts):
        """terms: one or two (x [N,C,H,W], m [N,C], a [N,H,W], b [N,H,W]) float32 tuples -> bf16 [parts, N, H, W, c_pad] =
        split(sum_t x_t * a_t + m_t * b_t); see pgpp_mix_pack"""
        lib = load_library()
        _torch_check(len(terms) in (1, 2), 'mix_pack takes one or two terms')
        x0 = terms[0][0]
        n, c, h, w = x0.shape
        flat = []
        for x, m, a, b in terms:
            _torch_check(x.is_cuda and x.dtype == torch.float32 and tuple(x.shape) == (n, c, h, w), 'mix_pack: x must be float32 [N,C,H,W]')
            flat += [x.contiguous(), m.to(torch.float32).reshape(n, c).contiguous(), a.to(torch.float32).reshape(n, h, w).contiguous(),
                     b.to(torch.float32).reshape(n, h, w).contiguous()]
        ptrs = [_ptr(t) for t in flat] + [None] * (8 - len(flat))
        out = torch.empty([parts, n, h, w, c_pad], dtype=torch.bfloat16, device=x0.device)
        with torch.cuda.device(x0.device):
            _check(lib.pgpp_mix_pack(*ptrs, _ptr(out), n, c, h, w, int(c_pad), int(parts), _stream(x0)))
        return out

    @staticmethod
    def conv2d_igemm(desc, device):
        lib = load_library()
        with torch.cuda.device(device):
            stream = ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
            _check(lib.pgpp_conv2d_igemm(ctypes.byref(desc), stream))

    @staticmethod
    def conv2d_igemm_stats_rows(desc, device):
        """rows of the instance-norm partial workspace this launch would fill (0: it cannot produce statistics)"""
        lib = load_library()
        with torch.cuda.device(device):
            rows = int(lib.pgpp_conv2d_igemm_stats_rows(ctypes.byref(desc)))
        if rows < 0:
            raise RuntimeError(lib.pgpp_last_error().decode())
        return rows

    @staticmethod
    def instnorm_finalize(ws, n, eps):
        """ws float32 [3, rows, C] (warp partials written by conv2d_igemm) -> (mean [N, C], rstd [N, C]) float32"""
        lib = load_library()
        rows, c = int(ws.shape[1]), int(ws.shape[2])
        mean = torch.empty([n, c], dtype=torch.float32, device=ws.device)
        rstd = torch.empty([n, c], dtype=torch.float32, device=ws.device)
        with torch.cuda.device(ws.device):
            _check(lib.pgpp_instnorm_finalize(_ptr(ws), rows, int(n), c, float(eps), _ptr(mean), _ptr(rstd), _stream(ws)))
        return mean, rstd

    @staticmethod
    def conv2d_wgrad(desc, device):
        lib = load_library()
        with torch.cuda.device(device):
            stream = ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
            _check(lib.pgpp_conv2d_wgrad(ctypes.byref(desc), stream))


class _IoEdgePlugin:
    """input / output edge of the inference loop (test.py:126-147, :162-166)"""

    @staticmethod
    def u8_to_f32(src, dst, c_off=0, normalize=True, mask=None):
        """src uint8 [N,C,H,W] -> channels [c_off, c_off+C) of dst float32 [N,Ct,H,W]; see pgpp_u8_to_f32"""
        _torch_check(src.is_cuda and src.dtype == torch.uint8 and src.dim() == 4 and src.is_contiguous(), 'src must be a contiguous uint8 CUDA tensor [N,C,H,W]')
        _torch_check(dst.is_cuda and dst.dtype == torch.float32 and dst.dim() == 4 and dst.is_contiguous() and dst.device == src.device,
                     'dst must be a contiguous float32 CUDA tensor on the same device')
        n, c, h, w = src.shape
        _torch_check(dst.shape[0] == n and tuple(dst.shape[2:]) == (h, w) and 0 <= c_off and c_off + c <= dst.shape[1], 'dst does not hold the channel slice')
        if mask is not None:
            _torch_check(mask.is_cuda and mask.dtype == torch.float32 and mask.is_contiguous() and tuple(mask.shape) == (n, 1, h, w),
                         'mask must be a contiguous float32 tensor [N,1,H,W]')
        lib = load_library()
        if src.numel() == 0:
            return dst
        with torch.cuda.device(src.device):
            _check(lib.pgpp_u8_to_f32(_ptr(src), n, c, h * w, _ptr(dst), dst.shape[1], int(c_off), int(bool(normalize)), _ptr(mask), _stream(src)))
        return dst

    @staticmethod
    def image_to_u8(img, reverse_channels=True):
        """img float32 [N,C,H,W] -> uint8 [N,H,W,C]; see pgpp_image_to_u8"""
        _torch_check(img.is_cuda and img.dtype == torch.float32 and img.dim() == 4 and img.is_contiguous(), 'img must be a contiguous float32 CUDA tensor [N,C,H,W]')
        n, c, h, w = img.shape
        out = torch.empty([n, h, w, c], dtype=torch.uint8, device=img.device)
        lib = load_library()
        if img.numel() == 0:
            return out
        with torch.cuda.device(img.device):
            _check(lib.pgpp_image_to_u8(_ptr(img), n, c, h * w, _ptr(out), int(bool(reverse_channels)), _stream(img)))
        return out


class _GridSamplePlugin:
    """aten::grid_sampler_2d / grid_sampler_2d_backward with (bilinear, zeros, align_corners=False), the only mode the reference
    uses (grid_sample_gradfix.py:49,64-65)"""

    @staticmethod
    def _check_operands(input, grid):
        _torch_check(input.is_cuda and grid.is_cuda and input.device == grid.device, 'input and grid must reside on the same CUDA device')
        _torch_check(input.dtype == torch.float32 and grid.dtype == torch.float32, 'grid_sample: float32 tensors only')
        _torch_check(input.dim() == 4 and grid.dim() == 4 and grid.shape[3] == 2 and grid.shape[0] == input.shape[0],
                     'grid_sample: input [N,C,H,W], grid [N,Ho,Wo,2]')
        _torch_check(input.shape[2] >= 1 and input.shape[3] >= 1, 'grid_sample: input must be at least 1x1')

    @staticmethod
    def forward(input, grid):
        _GridSamplePlugin._check_operands(input, grid)
        lib = load_library()
        input, grid = input.contiguous(), grid.contiguous()
        n, c, h, w = input.shape
        ho, wo = grid.shape[1], grid.shape[2]
        out = torch.empty([n, c, ho, wo], dtype=torch.float32, device=input.device)
        with torch.cuda.device(input.device):
            _check(lib.pgpp_grid_sample_2d(_ptr(input), _ptr(grid), _ptr(out), n, c, h, w, ho, wo, _stream(input)))
        return out

    @staticmethod
    def backward(grad_output, input, grid, need_input=True, need_grid=True):
        _GridSamplePlugin._check_operands(input, grid)
        lib = load_library()
        grad_output, input, grid = grad_output.to(torch.float32).contiguous(), input.contiguous(), grid.contiguous()
        n, c, h, w = input.shape
        ho, wo = grid.shape[1], grid.shape[2]
        _torch_check(tuple(grad_output.shape) == (n, c, ho, wo), 'grid_sample backward: grad_output has the wrong shape')
        gi = torch.empty_like(input) if need_input else None
        gg = torch.empty_like(grid) if need_grid else None
        if need_input or need_grid:
            with torch.cuda.device(input.device):
                _check(lib.pgpp_grid_sample_2d_backward(_ptr(grad_output), _ptr(input), _ptr(grid), _ptr(gi), _ptr(gg), n, c, h, w, ho, wo,
                                                        _stream(input)))
        return gi, gg


_PLUGINS = {'bias_act_plugin': _BiasActPlugin, 'upfirdn2d_plugin': _Upfirdn2dPlugin, 'conv2d_plugin': _ConvPlugin,
            'io_edge_plugin': _IoEdgePlugin, 'grid_sample_plugin': _GridSamplePlugin}


def get_plugin(module_name, sources=None, **build_kwargs):
    """Same call shape as the reference (`sources` / build kwargs are accepted and ignored: nothing is compiled)."""
    assert verbosity in ['none', 'brief', 'full']
    if module_name in _cached_plugins:
        return _cached_plugins[module_name]
    if module_name not in _PLUGINS:
        raise RuntimeError(f'unknown plugin "{module_name}"; available: {sorted(_PLUGINS)}')
    load_library()
    if verbosity == 'full':
        print(f'Loaded prebuilt PyTorch plugin "{module_name}" from {_LIB_PATH}')
    _cached_plugins[module_name] = _PLUGINS[module_name]
    return _cached_plugins[module_name]
