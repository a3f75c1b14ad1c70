"""CPU tests (-m "not gpu"): the launch plan of the implicit-GEMM convolution (pgpp_conv2d_igemm_plan) as a pure function of the
descriptor - which MMA issuer, weight residency, stacking, channel block, epilogue and statistics rows a launch gets on a 148-SM B200 -
and the coverage of the GPU issuer matrix (tests/igemm_matrix.py) over every leaf of the issuer ladder."""
import ctypes
import itertools

import pytest

from igemm_matrix import ALL_LEAVES, CASE, ISSUER_CASES, case_desc, cg, custom_ops, issuer_leaf, leaf_is_resident, switches

BF16, F32, E4M3 = 2, 0, 4


def plan_of(d):
    cg._init()
    return cg._plugin.conv2d_igemm_plan(d)


def test_gpu_matrix_names_every_issuer_leaf():
    named = [c[0] for c in ISSUER_CASES]
    assert len(ALL_LEAVES) == 33 and len(named) == len(set(named))
    assert set(named) == ALL_LEAVES, set(named) ^ ALL_LEAVES


@pytest.mark.parametrize('case', ISSUER_CASES, ids=[c[0] for c in ISSUER_CASES])
def test_case_plans_to_its_leaf(case):
    with switches(case[9]):
        p = plan_of(case_desc(case))
    assert issuer_leaf(p) == case[0], p
    assert p['grid'] == min(p['total_tiles'], 148) and p['tw'] * p['th'] * p['tn'] == 128


# leaf, b_resident, stack, kb, epilogue, stats_rows (float32 NCHW output: the general epilogue; statistics need whole pixel tiles)
PINNED = [
    ('slab i9 p2 stk', 1, 1, 64, 0, 8 * 4 * 6 * 4),
    ('slab i9 p2', 1, 0, 64, 0, 0),              # 61 x 67: ragged tiles, no statistics
    ('slab9 p2', 1, 0, 64, 0, 8 * 4 * 6 * 4),
    ('i3 p2 stk', 1, 1, 64, 0, 0),               # 15 rows: not whole 8-row tiles
    ('i3 p2 res', 1, 0, 64, 0, 0),               # 10 rows: not whole 8-row tiles
    ('i3 p2', 0, 0, 64, 0, 4 * 8 * 10 * 4),
    ('i3 p3', 0, 0, 64, 0, 0),
    ('i1 p2 res', 1, 0, 64, 0, 0),               # 96 columns in 128-pixel rows
    ('generic res', 1, 0, 64, 0, 0),
    ('f8 i3 res', 1, 0, 128, 0, 4 * 8 * 6 * 4),
    ('f8 generic res', 1, 0, 64, 0, 0),
    ('f8 i7', 0, 0, 128, 0, 2 * 4),              # two 16 x 8 tiles, four warp partials each
]


@pytest.mark.parametrize('leaf,res,stack,kb,epi,rows', PINNED, ids=[c[0] for c in PINNED])
def test_exact_plan(leaf, res, stack, kb, epi, rows):
    case = CASE[leaf]
    with switches(case[9]):
        p = plan_of(case_desc(case))
    assert (issuer_leaf(p), p['b_resident'], p['stack'], p['kb'], p['epilogue'], p['stats_rows']) == (leaf, res, stack, kb, epi, rows), p


def _packed_out(d, parts=1, e4m3=False):
    """turn a case descriptor into one that writes the channels-innermost operand format"""
    c_tot = d.o
    d.out_dtype = E4M3 if e4m3 else BF16
    d.out_stride = (ctypes.c_int64 * 4)(d.conv_h * d.conv_w * c_tot, 1, d.conv_w * c_tot, c_tot)
    d.out_parts = parts
    d.out_part_stride = d.n * d.conv_h * d.conv_w * c_tot
    return d


def test_epilogue_selection():
    d = _packed_out(case_desc(CASE['slab i9 p2 stk']), parts=2)
    assert plan_of(d)['epilogue'] == 1 and plan_of(d)['stack'] == 1
    with switches(('PGPP_IGEMM_NO_LEAN_EPILOGUE',)):
        assert plan_of(d)['epilogue'] == 0
    d.act_fn = 4                                    # tanh: gain not foldable -> general epilogue, no stacking, not fast
    p = plan_of(d)
    assert (p['epilogue'], p['stack'], p['fast'], issuer_leaf(p)) == (0, 0, 0, 'slab i9 p2')
    d = _packed_out(case_desc(CASE['f8 slab inner9']), e4m3=True)
    assert plan_of(d)['epilogue'] == 1
    d.out_parts = 2
    with pytest.raises(RuntimeError, match='split output needs bf16'):
        plan_of(d)


@pytest.mark.parametrize('name,field,value', [
    ('PGPP_IGEMM_NO_REUSE', 'reuse', 0), ('PGPP_IGEMM_NO_SLAB2', 'reuse', 1), ('PGPP_IGEMM_NO_RESIDENT', 'b_resident', 0),
    ('PGPP_IGEMM_NO_STACK', 'stack', 0)])
def test_switches_take_effect(name, field, value):
    d = case_desc(CASE['slab i9 p2 stk'])
    assert plan_of(d)[field] != value
    with switches((name,)):
        assert plan_of(d)[field] == value


def test_plan_needs_no_device_and_validates():
    lib = custom_ops.load_library()
    plan = custom_ops.IgemmPlan()
    assert lib.pgpp_conv2d_igemm_plan(ctypes.byref(case_desc(ISSUER_CASES[0])), None) != 0
    assert 'NULL' in lib.pgpp_last_error().decode()
    d = case_desc(ISSUER_CASES[0])
    d.block_n = 48
    assert lib.pgpp_conv2d_igemm_plan(ctypes.byref(d), ctypes.byref(plan)) != 0 and 'block_n' in lib.pgpp_last_error().decode()


@pytest.mark.parametrize('c_pad,e4m3,kb', [(16, False, 16), (32, False, 32), (48, False, 16), (32, True, 32), (64, True, 64), (96, True, 32)])
def test_narrow_channel_blocks(c_pad, e4m3, kb):
    """channel widths the Python packers never produce (they pad to 64): smaller K blocks with 32- / 64-byte swizzle rows, generic issuer"""
    d = case_desc(CASE['f8 generic' if e4m3 else 'generic'])
    d.c_pad = d.act_pixel_stride = c_pad
    p = plan_of(d)
    assert p['kb'] == kb and issuer_leaf(p) == ('f8 generic' if e4m3 else 'generic'), p
    if e4m3 and c_pad == 32:
        d.c_pad = d.act_pixel_stride = 48
        with pytest.raises(RuntimeError, match='multiple of 32'):
            plan_of(d)


def test_resident_weights_only_on_issuers_that_read_them():
    """every plan with resident weights dispatches to a resident issuer and vice versa: an issuer that waits on the weight ring while the
    producer loaded the weights once (or the reverse) would stall at its second tile"""
    bad = []
    for prec, k, o, ic, (n, h, w) in itertools.product(('bf16', 'bf16x2', 'bf16x3', 'fp8'), (1, 2, 3, 5, 7), (16, 32, 64, 128, 256),
                                                         (32, 64, 128, 192), ((1, 16, 16), (2, 40, 40), (6, 64, 64), (4, 100, 100), (10, 12, 128))):
        case = ('?', n, ic, o, k, h, w, k // 2, prec, ())
        for env in ((), ('PGPP_IGEMM_NO_REUSE',), ('PGPP_IGEMM_SLAB9',)):
            with switches(env):
                try:
                    p = plan_of(case_desc(case))
                except RuntimeError:
                    continue
            if leaf_is_resident(issuer_leaf(p)) != bool(p['b_resident']):
                bad.append((case, env, issuer_leaf(p), p['b_resident']))
    assert not bad, bad[:10]
