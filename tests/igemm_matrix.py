"""The MMA-issuer ladder of csrc/conv_igemm.cu and a launch matrix that reaches every leaf of it.

Shared by the CPU pins of the launch plan (test_igemm_plan_cpu.py) and the GPU numerics (test_gpu_p_igemm_paths.py): the CPU test
asserts that every case below plans to the leaf it names and that the cases name all leaves, the GPU test runs them."""
import contextlib
import ctypes
import importlib
import os

from conftest import load_pkg

load_pkg()
cg = importlib.import_module('pgpp_b200.torch_utils.ops.conv2d_gradfix')
custom_ops = importlib.import_module('pgpp_b200.torch_utils.custom_ops')

SMS = 148       # B200


def issuer_leaf(p):
    """The issuer a launch plan dispatches to: a mirror of the ladder in igemm_kernel (csrc/conv_igemm.cu:1064-1095)."""
    res, inner, parts, stk = p['b_resident'], p['inner'], p['parts'], p['stack']
    if p['e4m3']:
        ks4 = p['kb'] == 128
        if p['reuse'] == 2:
            return 'f8 slab9' if p['slab9'] else ('f8 slab inner9' if inner == 9 else 'f8 slab generic')
        if ks4 and inner == 3:
            return 'f8 i3 res' if res else 'f8 i3'
        if ks4 and inner == 7:
            return 'f8 i7'
        if ks4 and inner == 1:
            return 'f8 i1 res' if res else 'f8 i1'
        return 'f8 generic res' if res else 'f8 generic'
    ks4 = p['kb'] == 64
    if p['reuse'] == 2 and p['slab9']:
        return 'slab9 p1' if parts == 1 else ('slab9 p2 stk' if stk else 'slab9 p2')
    if p['reuse'] == 2:
        if inner == 9 and parts == 1:
            return 'slab i9 p1'
        if inner == 9 and parts == 2:
            return 'slab i9 p2 stk' if stk else 'slab i9 p2'
        return 'slab stk' if stk else 'slab generic'
    if ks4 and inner == 3 and parts == 1:
        return 'i3 p1 res' if res else 'i3 p1'
    if ks4 and inner == 3 and parts == 2 and stk:
        return 'i3 p2 stk'
    if ks4 and inner == 1 and parts == 2 and stk:
        return 'i1 p2 stk'
    if ks4 and inner == 3 and parts == 2:
        return 'i3 p2 res' if res else 'i3 p2'
    if ks4 and inner == 3 and parts == 3:
        return 'i3 p3'
    if ks4 and inner == 7 and parts in (1, 2):
        return f'i7 p{parts}'
    if ks4 and inner == 1 and parts in (1, 2):
        return f'i1 p{parts} res' if res else f'i1 p{parts}'
    return 'generic res' if res else 'generic'


ALL_LEAVES = frozenset([
    'slab9 p1', 'slab9 p2 stk', 'slab9 p2', 'slab i9 p1', 'slab i9 p2 stk', 'slab i9 p2', 'slab stk', 'slab generic',
    'i3 p1 res', 'i3 p1', 'i3 p2 stk', 'i1 p2 stk', 'i3 p2 res', 'i3 p2', 'i3 p3', 'i7 p1', 'i7 p2',
    'i1 p1 res', 'i1 p1', 'i1 p2 res', 'i1 p2', 'generic res', 'generic',
    'f8 slab9', 'f8 slab inner9', 'f8 slab generic', 'f8 i3 res', 'f8 i3', 'f8 i7', 'f8 i1 res', 'f8 i1', 'f8 generic res', 'f8 generic'])


def leaf_is_resident(leaf):
    """whether the issuer reads its weights from resident slots (as opposed to waiting on the weight ring)"""
    return 'res' in leaf or 'stk' in leaf or 'slab' in leaf


SLAB9 = ('PGPP_IGEMM_SLAB9',)
# leaf, n, ic, o, k, h, w, pad, precision, switches.  Between them: ragged tiles (odd sizes), padding 0 and k - 1, two or more channel
# blocks (ic 100 / 128 / 192 / 256), ic not a multiple of 64, and more than 2 x 148 tiles on a resident and on a ring leaf
# ('i1 p2 res', 'i3 p2': every CTA reuses both accumulator buffers and wraps its rings).
ISSUER_CASES = [
    ('slab i9 p1', 6, 64, 32, 3, 64, 64, 1, 'bf16', ()),
    ('slab i9 p2', 6, 100, 32, 3, 61, 67, 1, 'bf16x2', ()),
    ('slab i9 p2 stk', 6, 64, 64, 3, 64, 64, 1, 'bf16x2', ()),
    ('slab generic', 6, 64, 32, 2, 48, 48, 1, 'bf16', ()),
    ('slab stk', 6, 64, 64, 2, 48, 48, 1, 'bf16x2', ()),
    ('slab9 p1', 6, 64, 64, 3, 64, 64, 1, 'bf16', SLAB9),
    ('slab9 p2 stk', 6, 64, 64, 3, 64, 64, 1, 'bf16x2', SLAB9),
    ('slab9 p2', 6, 64, 64, 3, 64, 64, 1, 'bf16x2', SLAB9 + ('PGPP_IGEMM_NO_STACK',)),
    ('i3 p1 res', 6, 64, 128, 3, 64, 64, 1, 'bf16', ()),
    ('i3 p1', 2, 64, 64, 3, 32, 32, 1, 'bf16', ()),
    ('i3 p2 stk', 10, 64, 64, 3, 15, 128, 1, 'bf16x2', ()),
    ('i3 p2 res', 10, 64, 32, 3, 10, 128, 1, 'bf16x2', ()),
    ('i3 p2', 10, 64, 256, 3, 64, 64, 1, 'bf16x2', ()),
    ('i3 p3', 2, 128, 64, 3, 20, 36, 0, 'bf16x3', ()),
    ('i7 p1', 1, 64, 32, 7, 16, 16, 3, 'bf16', ()),
    ('i7 p2', 1, 64, 32, 7, 22, 19, 6, 'bf16x2', ()),
    ('i1 p1 res', 2, 64, 32, 1, 96, 96, 0, 'bf16', ()),
    ('i1 p1', 2, 192, 64, 1, 16, 16, 0, 'bf16', ()),
    ('i1 p2 res', 4, 64, 32, 1, 96, 96, 0, 'bf16x2', ()),
    ('i1 p2 stk', 2, 64, 64, 1, 96, 96, 0, 'bf16x2', ()),
    ('i1 p2', 2, 128, 64, 1, 17, 15, 0, 'bf16x2', ()),
    ('generic res', 2, 64, 32, 1, 96, 96, 0, 'bf16x3', ()),
    ('generic', 2, 64, 32, 5, 16, 16, 2, 'bf16x2', ()),
    ('f8 slab9', 6, 128, 64, 3, 64, 64, 1, 'fp8', SLAB9),
    ('f8 slab inner9', 6, 128, 32, 3, 64, 64, 1, 'fp8', ()),
    ('f8 slab generic', 6, 128, 32, 2, 48, 48, 1, 'fp8', ()),
    ('f8 i3 res', 6, 128, 128, 3, 64, 64, 1, 'fp8', ()),
    ('f8 i3', 2, 256, 64, 3, 33, 31, 1, 'fp8', ()),
    ('f8 i7', 1, 128, 32, 7, 16, 16, 3, 'fp8', ()),
    ('f8 i1 res', 2, 128, 32, 1, 96, 96, 0, 'fp8', ()),
    ('f8 i1', 2, 256, 64, 1, 16, 16, 0, 'fp8', ()),
    ('f8 generic res', 2, 64, 32, 1, 96, 96, 0, 'fp8', ()),
    ('f8 generic', 2, 64, 32, 3, 32, 32, 1, 'fp8', ()),
]
CASE = {c[0]: c for c in ISSUER_CASES}


@contextlib.contextmanager
def switches(names):
    """set PGPP_* switches (value 1) for the duration of the block; the library re-reads them on entry and exit"""
    saved = {k: os.environ.get(k) for k in names}
    for k in names:
        os.environ[k] = '1'
    custom_ops.refresh_env()
    try:
        yield
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        custom_ops.refresh_env()


def case_desc(case, out_dtype=0):
    """pgpp_conv_desc of the launch igemm_conv makes for a case on a PackedAct input with float32 NCHW output, on dummy pointers
    (planning never dereferences them)"""
    _, n, ic, o, k, h, w, pad, prec, _ = case
    products, parts = cg._PRODUCTS[prec]
    phase_stride, cols, o_rows, c_pad = cg.weight_layout(o, ic)
    conv_h, conv_w = h + 2 * pad - k + 1, w + 2 * pad - k + 1
    tw = min(128, 1 << (conv_w - 1).bit_length())
    th = min(128 // tw, 1 << (conv_h - 1).bit_length())
    m_tiles = -(-conv_w // tw) * -(-conv_h // th) * -(-n // (128 // (tw * th)))
    block_n = cg.choose_block_n(cols, m_tiles)
    while o_rows % block_n:
        block_n //= 2
    d = custom_ops.ConvDesc()
    d.act = d.wgt = d.out = 0x10000
    d.a_parts = d.b_parts = parts
    d.n, d.h, d.w, d.c_pad, d.act_pixel_stride = n, h, w, c_pad, c_pad
    d.kh = d.kw = k
    d.pad_y = d.pad_x = pad
    d.stride, d.dil_y = 1, 1
    d.conv_h, d.conv_w = conv_h, conv_w
    d.o, d.phases, d.phase_stride, d.o_rows, d.block_n, d.products = o, 1, phase_stride, o_rows, block_n, products
    d.act_fn, d.gain, d.clamp = 1, 1.0, -1.0
    d.out_dtype, d.out_h, d.out_w = out_dtype, conv_h, conv_w
    d.out_stride = (ctypes.c_int64 * 4)(o * conv_h * conv_w, conv_h * conv_w, conv_w, 1)
    d.out_parts = 1
    if prec == 'fp8':
        d.operand_e4m3, d.wscale = 1, 0x10000
    return d
