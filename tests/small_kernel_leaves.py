"""The kernel instantiations of csrc/conv_pack.cu, fir_packed.cu, conv_thin.cu and reduce.cu, and the launch cases that reach each.

Shared by the CPU inventory (test_small_kernel_leaves_cpu.py: the library holds exactly these instantiations) and the GPU numerics
(test_gpu_q_small_kernel_paths.py: every case runs, records the kernels it launched and checks the one it names).  Plain data: no torch.

A leaf name is the kernel's name without namespace, return type and parameter list, template arguments without casts and spaces,
booleans as 1 / 0: `mul_reduce_kernel<256>`.  `leaf_name` derives it from a cu++filt symbol and from a profiler kernel name alike."""
import re

# the kernels defined in the four files (upfirdn2d.cu has a fir_tile_kernel, hence exact names)
KERNELS = frozenset([
    'pack_nchw_kernel', 'pack_generic_kernel', 'im2col_kernel', 'spade_pack_kernel', 'conv_direct_kernel', 'fir_pack_kernel',
    'mix_pack_kernel', 'demod_kernel', 'modulate_weights_kernel',                                   # conv_pack.cu
    'fir_packed_kernel', 'fir_tile_packed_kernel', 'copy_packed_kernel',                            # fir_packed.cu
    'conv1x1_thin_kernel',                                                                          # conv_thin.cu
    'mul_reduce_kernel', 'sum_hw_kernel',                                                           # reduce.cu
])

_CAST = re.compile(r'\((?:unsigned )?(?:int|bool|long long|long|char)\)')


def leaf_name(symbol):
    """'void pgpp::mul_reduce_kernel<(int)256>(pgpp::MulReduceArgs)' / 'pgpp::mul_reduce_kernel<256>(...)' -> 'mul_reduce_kernel<256>'"""
    s = _CAST.sub('', symbol)
    s = re.sub(r'\btrue\b', '1', s)
    s = re.sub(r'\bfalse\b', '0', s)
    s = s.strip()
    if s.startswith('void '):
        s = s[5:]
    depth = 0
    for i, ch in enumerate(s):           # the parameter list starts at the first '(' outside the template argument list
        if ch == '<':
            depth += 1
        elif ch == '>':
            depth -= 1
        elif ch == '(' and depth == 0:
            s = s[:i]
            break
    s = s.replace(' ', '')
    return s[len('pgpp::'):] if s.startswith('pgpp::') else s


def base_name(leaf):
    return leaf.split('<', 1)[0]


F32, F16, BF16, F64 = 'float', '__half', '__nv_bfloat16', 'double'

# ---- pgpp_pack_activations* -------------------------------------------------------------------------------------------------
# (leaf, source dtype, (n, c, h, w), view, mode, c_slice)
#   view: 'contig' | 'pitch' (row pitch w + 4, or the next multiple of 4) | 'misaligned' (base 1 element off) | 'sn_odd' (sample
#         stride not a multiple of 4) | 'cl' (channels_last) | 'step2' ([..., ::2])
#   mode: 1 / 2 / 3 bf16 parts, 'f16' (one IEEE half part), 'e4m3' (one byte part)
#   c_slice: None, or (c_total, c_off) of a wider destination whose other channels must stay untouched
PACK_CASES = [
    ('pack_nchw_kernel<float,1,0>', F32, (2, 64, 16, 128), 'contig', 2, None),
    ('pack_nchw_kernel<float,1,0>', F32, (1, 70, 8, 64), 'contig', 3, None),
    ('pack_nchw_kernel<float,1,0>', F32, (2, 24, 5, 32), 'contig', 1, (192, 64)),
    ('pack_nchw_kernel<float,1,0>', F32, (1, 8, 9, 130), 'pitch', 2, None),
    ('pack_nchw_kernel<float,1,0>', F32, (2, 16, 6, 16), 'pitch', 'e4m3', None),
    ('pack_nchw_kernel<__half,1,0>', F16, (2, 64, 16, 64), 'contig', 2, None),
    ('pack_nchw_kernel<__half,1,0>', F16, (1, 70, 4, 32), 'contig', 'f16', (160, 80)),
    ('pack_nchw_kernel<__nv_bfloat16,1,0>', BF16, (1, 70, 9, 32), 'contig', 3, None),
    ('pack_nchw_kernel<__nv_bfloat16,1,0>', BF16, (2, 8, 3, 16), 'pitch', 2, (136, 8)),
    ('pack_nchw_kernel<float,0,0>', F32, (2, 24, 7, 7), 'contig', 2, None),
    ('pack_nchw_kernel<float,0,0>', F32, (1, 70, 5, 33), 'contig', 3, (144, 0)),
    ('pack_nchw_kernel<float,0,0>', F32, (2, 16, 4, 32), 'misaligned', 2, None),
    ('pack_nchw_kernel<float,0,0>', F32, (3, 8, 4, 16), 'sn_odd', 1, None),
    ('pack_nchw_kernel<float,0,0>', F32, (1, 16, 5, 13), 'contig', 'e4m3', None),
    ('pack_nchw_kernel<__half,0,0>', F16, (2, 24, 7, 7), 'contig', 2, None),
    ('pack_nchw_kernel<__half,0,0>', F16, (1, 16, 3, 130), 'misaligned', 'f16', None),
    ('pack_nchw_kernel<__nv_bfloat16,0,0>', BF16, (1, 70, 5, 33), 'contig', 2, (208, 64)),
    ('pack_nchw_kernel<double,0,0>', F64, (2, 24, 8, 16), 'contig', 2, None),
    ('pack_nchw_kernel<double,0,0>', F64, (1, 70, 3, 130), 'contig', 3, (160, 16)),
    ('pack_generic_kernel<float>', F32, (2, 70, 6, 10), 'cl', 2, None),
    ('pack_generic_kernel<float>', F32, (1, 24, 5, 9), 'step2', 3, (96, 32)),
    ('pack_generic_kernel<__half>', F16, (2, 24, 5, 7), 'cl', 2, None),
    ('pack_generic_kernel<__nv_bfloat16>', BF16, (1, 40, 4, 6), 'cl', 1, (128, 64)),
    ('pack_generic_kernel<double>', F64, (2, 24, 5, 7), 'cl', 3, None),
    ('pack_generic_kernel<double>', F64, (1, 16, 4, 8), 'step2', 'e4m3', None),
]

# ---- pgpp_pack_act_gradient (pack_nchw_kernel<T, VEC, true>) ------------------------------------------------------------------
# (leaf, dtype, (n, c, h, w), act, alpha, gain, clamp, mode)   w % 4 != 0 takes the element-load form
ACT_GRAD_CASES = [
    ('pack_nchw_kernel<float,1,1>', F32, (2, 24, 40, 36), 'lrelu', 0.25, 1.5, 3.0, 2),
    ('pack_nchw_kernel<float,1,1>', F32, (1, 70, 8, 64), 'relu', 0.0, -2.0, -1.0, 3),
    ('pack_nchw_kernel<float,0,1>', F32, (2, 24, 9, 7), 'linear', 0.0, -0.5, 3.0, 2),
    ('pack_nchw_kernel<float,0,1>', F32, (1, 16, 5, 33), 'lrelu', 0.25, -2.0, 3.0, 1),
    ('pack_nchw_kernel<__half,1,1>', F16, (2, 24, 16, 32), 'lrelu', 0.25, 2.0, 3.0, 'f16'),
    ('pack_nchw_kernel<__half,0,1>', F16, (1, 40, 7, 13), 'relu', 0.0, -1.5, 3.0, 2),
    ('pack_nchw_kernel<__nv_bfloat16,1,1>', BF16, (2, 24, 8, 16), 'lrelu', 0.25, -2.0, 3.0, 2),
    ('pack_nchw_kernel<__nv_bfloat16,0,1>', BF16, (1, 16, 9, 7), 'linear', 0.0, 1.5, 3.0, 1),
]

# ---- pgpp_pack_im2col: (leaf, dtype, (n, c, h, w), kw, r, pad_x, pad_y, scaled, parts) ----------------------------------------
IM2COL_CASES = [
    ('im2col_kernel<float>', F32, (2, 3, 10, 150), 7, 2, 3, 3, True, 3),
    ('im2col_kernel<float>', F32, (1, 1, 9, 40), 3, 4, 1, 0, False, 2),
    ('im2col_kernel<__half>', F16, (2, 6, 8, 140), 3, 2, 1, 1, True, 2),
    ('im2col_kernel<__nv_bfloat16>', BF16, (1, 3, 7, 33), 7, 1, 3, 2, False, 1),
    ('im2col_kernel<double>', F64, (2, 2, 6, 131), 5, 3, 2, 2, True, 3),
]

# ---- pgpp_spade_modulate_pack: (leaf, (n, c, h, w), c_pad, parts, pre_gain, gb_pad, x_offset) ----------------------------------
#   gb_pad: extra elements per sample between gamma / beta planes (2 breaks the 16-byte alignment of sample 1); x_offset: x misaligned
SPADE_CASES = [
    ('spade_pack_kernel<1>', (2, 64, 8, 32), 64, 2, 0.0, 0, 0),
    ('spade_pack_kernel<1>', (1, 70, 4, 16), 128, 3, 1.5, 0, 0),
    ('spade_pack_kernel<0>', (2, 24, 5, 7), 64, 2, 2.0, 0, 0),
    ('spade_pack_kernel<0>', (2, 16, 4, 16), 16, 1, 0.0, 2, 0),
    ('spade_pack_kernel<0>', (1, 16, 4, 32), 64, 2, 0.5, 0, 1),
]

# ---- pgpp_mix_pack: (leaf, (n, c, h, w), c_pad, parts, terms, misaligned) -----------------------------------------------------
MIX_CASES = [
    ('mix_pack_kernel<1>', (2, 64, 8, 32), 64, 2, 2, False),
    ('mix_pack_kernel<1>', (1, 70, 4, 16), 128, 3, 1, False),
    ('mix_pack_kernel<0>', (2, 24, 5, 7), 64, 2, 2, False),
    ('mix_pack_kernel<0>', (1, 16, 4, 16), 16, 1, 1, True),
]

# ---- pgpp_conv2d_direct: (leaf, n, c, h, w, o, kh, kw, act, clamp, packed) ------------------------------------------------------
#   packed: None (float32 NCHW) or (parts, c_total, c_off) of an operand-format destination
DIRECT_CASES = [
    ('conv_direct_kernel<3,3,1,2,0>', 2, 1, 33, 47, 64, 3, 3, 'relu', -1.0, None),
    ('conv_direct_kernel<3,3,1,2,0>', 1, 1, 17, 130, 72, 3, 3, 'relu', -1.0, (2, 144, 64)),
    ('conv_direct_kernel<3,3,1,0,1>', 2, 1, 20, 24, 64, 3, 3, 'lrelu', 2.5, None),
    ('conv_direct_kernel<3,3,1,0,1>', 1, 1, 9, 7, 8, 3, 3, 'relu', 2.5, (3, 72, 64)),
    ('conv_direct_kernel<1,1,0,0,1>', 2, 5, 40, 56, 64, 1, 1, 'lrelu', -1.0, None),
    ('conv_direct_kernel<1,1,0,0,1>', 1, 16, 9, 130, 72, 1, 1, 'linear', 2.5, (1, 80, 8)),
    ('conv_direct_kernel<1,0,0,0,1>', 2, 5, 20, 36, 64, 3, 1, 'lrelu', 2.5, None),
    ('conv_direct_kernel<1,0,0,0,1>', 1, 3, 17, 23, 24, 5, 1, 'relu', -1.0, (2, 88, 64)),
    ('conv_direct_kernel<1,0,0,0,1>', 2, 2, 33, 7, 16, 7, 1, 'linear', -1.0, None),
    ('conv_direct_kernel<3,0,0,0,1>', 2, 1, 21, 45, 64, 5, 3, 'lrelu', 2.5, None),
    ('conv_direct_kernel<3,0,0,0,1>', 1, 5, 16, 16, 16, 1, 3, 'relu', -1.0, (3, 80, 64)),
    ('conv_direct_kernel<3,0,0,0,1>', 1, 4, 13, 130, 8, 1, 3, 'linear', 2.5, None),
]

# ---- pgpp_modconv_demod_coefs: (leaf, n, o, i, kh, kw) -------------------------------------------------------------------------
DEMOD_CASES = [
    ('demod_kernel', 11, 24, 70, 3, 3),
    ('demod_kernel', 3, 8, 512, 1, 1),
    ('demod_kernel', 17, 5, 13, 3, 3),
]

# ---- pgpp_modulate_weights: (leaf, n, rows, c_pad, c_in, parts)   rows * c_pad / 8 > 4096 * 256: several grid-stride rounds --------
MODW_CASES = [
    ('modulate_weights_kernel', 2, 9 * 15000, 64, 50, 2),
    ('modulate_weights_kernel', 3, 9 * 40, 128, 128, 3),
    ('modulate_weights_kernel', 1, 7, 16, 3, 1),
]

# ---- pgpp_fir_pack (float32 NCHW -> operand format): (leaf, (n, c, h, w), taps (fh x fw, row-major), fh, fw, pad, flip, gain, parts)
FIR_PACK_CASES = [
    ('fir_pack_kernel', (2, 64, 32, 48), [1, 3, 3, 1, 3, 9, 9, 3, 3, 9, 9, 3, 1, 3, 3, 1], 4, 4, (2, 2, 2, 2), False, 0.25, 2),
    ('fir_pack_kernel', (1, 70, 17, 29), [1, -2, 3, 2, 0, 1], 3, 2, (1, 0, 1, 1), True, 2.0, 3),
]

# ---- pgpp_fir_packed / pgpp_fir_packed_act on the operand format ----------------------------------------------------------------
# (leaf, n, c, h, w, in_parts, out_parts, filter, down, pad (x0, x1, y0, y1), flip, gain, epilogue)
#   filter: 'sep121' (outer([1,2,1], [1,2,1])), 'sep1331', 'ns4x4' / 'ns3x2' (not separable), None (identity copy)
#   epilogue: None, or dict(noise='hw' | 'nhw' | None, bias, act, alpha, gain, clamp, nchw = c_out or None, dst_c_off)
_EPI = dict(noise='hw', bias=True, act='lrelu', alpha=0.25, gain=2.0, clamp=6.0, nchw=None, dst_c_off=0)
FIR_PACKED_CASES = [
    ('fir_packed_kernel<1,8>', 2, 72, 19, 23, 2, 2, 'ns4x4', 1, (2, 1, 1, 2), False, 0.5, None),
    ('fir_packed_kernel<1,8>', 1, 8, 13, 9, 3, 1, 'ns3x2', 1, (1, 0, 1, 1), True, 2.0, None),
    ('fir_packed_kernel<1,8>', 2, 16, 20, 6, 1, 3, 'ns4x4', 1, (1, 2, 2, 1), True, 1.0, None),
    ('fir_packed_kernel<2,4>', 2, 72, 19, 23, 2, 3, 'sep121', 2, (1, 1, 1, 1), False, 1.0, None),
    ('fir_packed_kernel<2,4>', 1, 8, 9, 9, 3, 1, 'ns3x2', 2, (1, 0, 0, 1), True, 2.0, None),
    ('fir_tile_packed_kernel<1,0>', 2, 72, 19, 23, 1, 2, 'sep121', 1, (1, 1, 1, 1), False, 1.0, None),
    ('fir_tile_packed_kernel<2,0>', 1, 8, 33, 17, 2, 2, 'sep1331', 1, (2, 2, 2, 2), True, 0.25, None),
    ('fir_tile_packed_kernel<3,0>', 2, 136, 16, 16, 3, 1, 'sep121', 1, (1, 1, 1, 1), False, 4.0, None),
    ('fir_tile_packed_kernel<1,1>', 2, 72, 19, 23, 1, 2, 'sep121', 1, (1, 1, 1, 1), False, 1.0, _EPI),
    ('fir_tile_packed_kernel<1,1>', 2, 8, 9, 17, 1, 1, 'sep121', 1, (1, 1, 1, 1), True, 0.5,
     dict(_EPI, noise='nhw', act='relu', clamp=-1.0, nchw=8)),
    ('fir_tile_packed_kernel<2,1>', 2, 72, 17, 25, 2, 2, 'sep1331', 1, (2, 2, 2, 2), False, 0.25,
     dict(_EPI, noise='nhw', act='linear', dst_c_off=64)),
    ('fir_tile_packed_kernel<2,1>', 1, 72, 12, 20, 2, 2, 'sep121', 1, (1, 1, 1, 1), False, 1.0, dict(_EPI, nchw=40)),
    ('fir_tile_packed_kernel<3,1>', 2, 8, 16, 8, 3, 3, 'sep121', 1, (1, 1, 1, 1), True, 1.0, dict(_EPI, noise=None, bias=False)),
    ('fir_tile_packed_kernel<3,1>', 1, 72, 9, 31, 3, 3, 'sep121', 1, (1, 1, 1, 1), False, 2.0, dict(_EPI, noise='hw', act='relu', nchw=72)),
    ('copy_packed_kernel', 2, 64, 16, 24, 2, 2, None, 1, (0, 0, 0, 0), False, 1.0, dict(dst_c_off=128)),
    ('copy_packed_kernel', 1, 72, 7, 9, 3, 3, None, 1, (0, 0, 0, 0), False, 1.0, dict(dst_c_off=8)),
]

# ---- pgpp_conv1x1_thin: (leaf, n, c, h, w, parts, o1, o2, c_off, accumulate1, act, clamp) ---------------------------------------
#   OT = 4 for o1 + o2 <= 4, else 8; LPP / CPL from c: <= 64 -> 8 / 1, <= 128 -> 16 / 1, <= 256 -> 32 / 1, else 32 / 2 (OT = 4 only)
THIN_CASES = []
for _parts in (1, 2, 3):
    THIN_CASES += [
        (f'conv1x1_thin_kernel<4,8,1,{_parts}>', 2, 8, 17, 19, _parts, 3, 0, 0, True, 'linear', -1.0),
        (f'conv1x1_thin_kernel<4,8,1,{_parts}>', 1, 64, 48, 48, _parts, 3, 1, 64, False, 'lrelu', 2.0),
        (f'conv1x1_thin_kernel<4,16,1,{_parts}>', 2, 72, 9, 31, _parts, 3, 1, 0, True, 'lrelu', 2.0),
        (f'conv1x1_thin_kernel<4,16,1,{_parts}>', 1, 128, 50, 50, _parts, 4, 0, 0, False, 'relu', -1.0),
        (f'conv1x1_thin_kernel<4,32,1,{_parts}>', 2, 200, 13, 11, _parts, 3, 0, 0, False, 'linear', 2.0),
        (f'conv1x1_thin_kernel<4,32,1,{_parts}>', 1, 256, 46, 47, _parts, 3, 1, 0, True, 'relu', -1.0),
        (f'conv1x1_thin_kernel<4,32,2,{_parts}>', 2, 512, 7, 23, _parts, 3, 0, 0, True, 'lrelu', 2.0),
        (f'conv1x1_thin_kernel<8,8,1,{_parts}>', 2, 64, 17, 19, _parts, 5, 0, 0, True, 'lrelu', 2.0),
        (f'conv1x1_thin_kernel<8,8,1,{_parts}>', 1, 8, 46, 47, _parts, 3, 5, 64, False, 'linear', -1.0),
        (f'conv1x1_thin_kernel<8,16,1,{_parts}>', 2, 72, 9, 31, _parts, 3, 5, 0, True, 'relu', 2.0),
        (f'conv1x1_thin_kernel<8,16,1,{_parts}>', 1, 128, 50, 50, _parts, 5, 0, 0, False, 'lrelu', -1.0),
        (f'conv1x1_thin_kernel<8,32,1,{_parts}>', 2, 200, 13, 11, _parts, 3, 5, 0, True, 'linear', 2.0),
        (f'conv1x1_thin_kernel<8,32,1,{_parts}>', 1, 256, 46, 47, _parts, 5, 0, 0, False, 'relu', -1.0),
    ]

# ---- pgpp_mul_reduce_hw / pgpp_sum_hw: G = 256 for hw >= 2048, else 32; float4 loads only for hw % 4 == 0 and 16-byte alignment ---
# mul_reduce: (leaf, n, c, hw, b, sub ('hw' | 'n1hw' | '11hw' | None), scale, out ('new' | 'alias' | None), misaligned)
MUL_REDUCE_CASES = [
    ('mul_reduce_kernel<32>', 2, 24, 720, True, 'hw', True, 'new', False),
    ('mul_reduce_kernel<32>', 3, 11, 2047, True, 'n1hw', True, 'alias', False),
    ('mul_reduce_kernel<32>', 2, 9, 720, True, None, True, 'new', True),
    ('mul_reduce_kernel<32>', 1, 5, 2046, False, None, False, None, False),
    ('mul_reduce_kernel<256>', 2, 6, 2048, True, 'hw', True, 'new', False),
    ('mul_reduce_kernel<256>', 2, 3, 512 * 512, True, '11hw', True, 'alias', False),
    ('mul_reduce_kernel<256>', 2, 4, 130 * 131, True, 'n1hw', True, 'new', False),
    ('mul_reduce_kernel<256>', 1, 5, 4096, True, None, True, 'new', True),
    ('mul_reduce_kernel<256>', 2, 3, 130 * 131, False, '11hw', False, None, False),
]
# sum_hw: (leaf, dtype, n, c, hw, misaligned)
SUM_HW_CASES = []
for _t in (F32, F16, BF16):
    SUM_HW_CASES += [
        (f'sum_hw_kernel<{_t},32>', _t, 2, 24, 720, False),
        (f'sum_hw_kernel<{_t},32>', _t, 3, 11, 2047, False),
        (f'sum_hw_kernel<{_t},32>', _t, 2, 9, 720, True),
        (f'sum_hw_kernel<{_t},256>', _t, 2, 6, 2048, False),
        (f'sum_hw_kernel<{_t},256>', _t, 1, 3, 512 * 512, False),
        (f'sum_hw_kernel<{_t},256>', _t, 2, 4, 130 * 131, False),
        (f'sum_hw_kernel<{_t},256>', _t, 1, 5, 4096, True),
    ]

FAMILIES = {
    'pack': PACK_CASES, 'act_grad': ACT_GRAD_CASES, 'im2col': IM2COL_CASES, 'spade': SPADE_CASES, 'mix': MIX_CASES,
    'direct': DIRECT_CASES, 'demod': DEMOD_CASES, 'modw': MODW_CASES, 'fir_pack': FIR_PACK_CASES, 'fir_packed': FIR_PACKED_CASES,
    'thin': THIN_CASES, 'mul_reduce': MUL_REDUCE_CASES, 'sum_hw': SUM_HW_CASES,
}

LEAVES = frozenset(case[0] for cases in FAMILIES.values() for case in cases)


def case_id(case):
    return '-'.join(str(v) for v in case if not isinstance(v, dict)).replace(' ', '')
