"""GPU tests: every MMA-issuer leaf and epilogue variant of the implicit-GEMM convolution (csrc/conv_igemm.cu) against an exact-product
float64 reference.

The reference reads the operands back from the packed buffers (bf16 parts of activations and weights, or e4m3 bytes times the weight
column scales) and computes in float64 exactly the products the precision mode runs, sum over pa + pb < parts of conv(A_pa, B_pb),
followed by the epilogue formula.  Only the kernel's fp32 accumulation separates the two, so a wrong tap, part, column tile or
sample shows up far above the tolerance.  Whether a launch dropped or added one whole split-precision product is checked separately
with operands of exactly one nonzero part each (test_product_set), where such a fault is an O(1) error.

Each case queries the launch plan of the launch it makes (pgpp_conv2d_igemm_plan) and asserts that it ran the issuer or epilogue it
names (on a 148-SM B200; other parts plan differently, and there only the numbers are checked)."""
import contextlib
import itertools
import math

import pytest
import torch
import torch.nn.functional as F

from helpers import rel_l2
from igemm_matrix import CASE, ISSUER_CASES, case_desc, cg, issuer_leaf, switches

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = 2e-5              # rel-L2 against the exact products: fp32 accumulation only
WORST = {}              # precision -> largest rel-L2 seen (printed by the last test, for the record)


def _b200():
    return torch.cuda.get_device_properties(0).multi_processor_count == 148


def assert_leaf(plan, leaf):
    if not _b200():
        pytest.skip(f'not a 148-SM B200 ({torch.cuda.get_device_name(0)}): the launch plans differently, leaf {leaf!r} not asserted '
                    '(numbers were checked)')
    assert issuer_leaf(plan) == leaf, plan


@contextlib.contextmanager
def plans():
    """the plans of every convolution launched in the block"""
    cg._init()
    seen, orig = [], cg._plugin.conv2d_igemm

    def launch(desc, device):
        with torch.cuda.device(device):
            seen.append(cg._plugin.conv2d_igemm_plan(desc))
        return orig(desc, device)
    cg._plugin.conv2d_igemm = launch
    try:
        yield seen
    finally:
        cg._plugin.conv2d_igemm = orig


def check_rounded(got, want, ulp, k=1.0):
    """a result rounded to a narrower type: at most k half-units in the last place (ulp = relative half-unit) plus the fp32
    accumulation (the exact-product tolerance, relative to the tensor's RMS)"""
    err = (got.double() - want).abs() - want.abs() * ulp * k
    assert float(err.max()) <= 4 * TOL * float(want.pow(2).mean().sqrt()) + 1e-7, float(err.max())


def check(got, want, prec, tol=TOL):
    e = rel_l2(got, want)
    WORST[prec] = max(WORST.get(prec, 0.0), e)
    assert e < tol, (prec, e)


def _randn(*shape, seed):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)).to(DEV)


def operands(case, seed=0, a_part=None, b_part=None):
    """(PackedAct, PackedWeights) of a case from the library's packers.  a_part / b_part: keep only that part of the activations /
    weights, filled with full-size bf16 values, and zero the others."""
    leaf, n, ic, o, k, h, w, pad, prec, _ = case
    parts = cg._PRODUCTS[prec][1]
    fp8 = prec == 'fp8'
    wt = _randn(o, ic, k, k, seed=seed) / math.sqrt(ic * k * k)
    pw = cg.pack_weights_native(wt, k, k, parts, pad, pad, e4m3=fp8)
    x = _randn(n, ic, h, w, seed=seed + 1)
    data = cg._plugin.pack_activations(x, None, pw.c_pad, parts, e4m3=fp8)
    if a_part is not None:
        full = data[0].clone()
        data.zero_()
        data[a_part] = full
    if b_part is not None:
        full = pw.data[0].clone()
        pw.data = torch.zeros_like(pw.data)
        pw.data[b_part] = full
    return cg.PackedAct(data, ic), pw


def gemm_ref(act, wgt, kh, kw, pad_y, pad_x, conv_h, conv_w, parts, wscale=None):
    """float64 sum over pa + pb < parts of conv(A_pa, B_pb): act [parts, N, H, W, C], wgt [parts, taps, cols, C] shared or
    [N, parts, taps, cols, C] per sample, wscale [cols] or [N, cols] (e4m3) -> GEMM columns [N, cols, conv_h, conv_w]"""
    a = act[:parts].double().permute(0, 1, 4, 2, 3)
    per_sample = wgt.dim() == 5
    out = 0
    for pa in range(parts):
        wsum = wgt[..., :parts - pa, :, :, :].double().sum(-4)         # [(N,) taps, cols, C]
        wk = wsum.reshape(*wsum.shape[:-3], kh, kw, wsum.shape[-2], wsum.shape[-1]).movedim(-2, -4).movedim(-1, -3)
        xp = F.pad(a[pa], [pad_x, kw, pad_y, kh])
        if per_sample:
            y = torch.cat([F.conv2d(xp[i:i + 1], wk[i]) for i in range(xp.shape[0])])
        else:
            y = F.conv2d(xp, wk)
        out = out + y[:, :, :conv_h, :conv_w]
    if wscale is not None:
        out = out * wscale.double().reshape(-1 if per_sample else 1, out.shape[1], 1, 1)
    return out


def case_ref(case, xp, pw, wgt=None, wscale=None):
    """float64 GEMM columns of a case's launch -> [N, o_rows, conv_h, conv_w]"""
    _, n, ic, o, k, h, w, pad, prec, _ = case
    parts = cg._PRODUCTS[prec][1]
    if wgt is None:
        wgt = pw.data if pw.data.dim() == 4 else pw.data[None]
        wscale = pw.wscale
    return gemm_ref(xp.data, wgt, k, k, pad, pad, h + 2 * pad - k + 1, w + 2 * pad - k + 1, parts, wscale)


def epilogue_ref(acc, dcoef=None, noise=None, bias=None, act='linear', alpha=0.2, gain=1.0, clamp=-1.0):
    r = acc.double()
    if dcoef is not None:
        r = r * dcoef.double()[:, :, None, None]
    if noise is not None:
        r = r + noise.double().reshape(-1 if noise.dim() == 4 else 1, 1, *noise.shape[-2:])
    if bias is not None:
        r = r + bias.double()[None, :, None, None]
    r = {'linear': r, 'relu': r.clamp_min(0), 'lrelu': torch.where(r < 0, r * alpha, r), 'tanh': torch.tanh(r)}[act] * gain
    return r.clamp(-clamp, clamp) if clamp >= 0 else r


def run(case, xp, pw, **kw):
    with switches(case[9]), plans() as seen:
        y = cg.igemm_conv(xp, pw, precision=case[8], **kw)
    torch.cuda.synchronize()
    assert len(seen) == 1
    return y, seen[0]


# ---- a. one case per issuer leaf -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize('case', ISSUER_CASES, ids=[c[0] for c in ISSUER_CASES])
def test_issuer_leaf(case):
    xp, pw = operands(case)
    y, plan = run(case, xp, pw, out_dtype=torch.float32)
    check(y, case_ref(case, xp, pw)[:, :case[3]], case[8])
    assert_leaf(plan, case[0])


@pytest.mark.parametrize('case', [('i7 p1', 10, 64, 16, 7, 12, 128, 3, 'bf16', ()), ('i3 p3', 6, 64, 16, 3, 64, 64, 1, 'bf16x3', ()),
                                  ('f8 i7', 10, 128, 16, 7, 12, 128, 3, 'fp8', ())], ids=['i7 p1', 'i3 p3', 'f8 i7'])
def test_ring_only_issuers_with_weights_that_fit(case):
    """16-column layers over more than 148 tiles whose weights would fit in shared memory, on issuers that only read the weight ring
    (images under 16 rows keep the 7 x 7 layers off the single-slab mode): the weights must be streamed (resident weights are loaded
    once, and these issuers would wait for a second ring phase)"""
    xp, pw = operands(case, seed=2)
    y, plan = run(case, xp, pw, out_dtype=torch.float32)
    check(y, case_ref(case, xp, pw)[:, :case[3]], case[8])
    assert plan['b_resident'] == 0 and plan['total_tiles'] > 148
    assert_leaf(plan, case[0])


# ---- b. the product set of every split-precision leaf ----------------------------------------------------------------------------

SPLIT = [c for c in ISSUER_CASES if cg._PRODUCTS[c[8]][1] > 1]


@pytest.mark.parametrize('case', SPLIT, ids=[c[0] for c in SPLIT])
def test_product_set(case):
    """exactly one nonzero part of A (i) and of B (j): the output is conv(A_i, B_j) when the mode runs that product (i + j < parts)
    and exactly zero when it does not"""
    parts = cg._PRODUCTS[case[8]][1]
    for i, j in itertools.product(range(parts), repeat=2):
        xp, pw = operands(case, seed=10 * i + j, a_part=i, b_part=j)
        y, plan = run(case, xp, pw, out_dtype=torch.float32)
        if i + j < parts:
            want = gemm_ref(xp.data[i:i + 1], pw.data[j:j + 1], case[4], case[4], case[7], case[7], y.shape[2], y.shape[3], 1)
            check(y, want[:, :case[3]], case[8])
        else:
            assert torch.count_nonzero(y) == 0, (i, j, float(y.abs().max()))
    assert_leaf(plan, case[0])


# ---- c. the epilogue variants on a stacked, an unstacked and an e4m3 leaf --------------------------------------------------------

EPI_LEAVES = ['slab i9 p2 stk', 'i3 p2 res', 'f8 slab inner9']


def _epi_args(case, noise_kind, seed=5):
    n, o = case[1], case[3]
    oh, ow = case[5] + 2 * case[7] - case[4] + 1, case[6] + 2 * case[7] - case[4] + 1
    noise = _randn(n, 1, oh, ow, seed=seed) if noise_kind == 'per_sample' else _randn(oh, ow, seed=seed)
    return dict(dcoef=_randn(n, o, seed=seed + 1).abs() + 0.5, noise=0.3 * noise, bias=0.5 * _randn(o, seed=seed + 2))


@pytest.mark.parametrize('leaf', EPI_LEAVES)
@pytest.mark.parametrize('out', ['f32', 'f32_channels_last', 'bf16', 'f16'])
def test_epilogue_tensor_output(leaf, out):
    case = CASE[leaf]
    xp, pw = operands(case, seed=3)
    ep = _epi_args(case, 'per_sample' if out == 'f32_channels_last' else 'plane')
    dt = {'f32': torch.float32, 'f32_channels_last': torch.float32, 'bf16': torch.bfloat16, 'f16': torch.float16}[out]
    mf = torch.channels_last if out == 'f32_channels_last' else torch.contiguous_format
    kw = dict(act='lrelu', alpha=0.2, gain=math.sqrt(2), clamp=1.5)
    y, plan = run(case, xp, pw, out_dtype=dt, memory_format=mf, **ep, **kw)
    want = epilogue_ref(case_ref(case, xp, pw)[:, :case[3]], **ep, **kw)
    if dt == torch.float32:
        check(y, want, case[8])
    else:               # one rounding to the output type: at most half a unit in the last place (and the fp32 accumulation)
        check_rounded(y, want, 2.0 ** (-8 if dt == torch.bfloat16 else -11))
    assert plan['epilogue'] == 0 and plan['fast'] == 1
    assert_leaf(plan, leaf)


@pytest.mark.parametrize('leaf', EPI_LEAVES)
@pytest.mark.parametrize('act', ['linear', 'relu', 'lrelu'])
@pytest.mark.parametrize('accumulate', [False, True])
@pytest.mark.parametrize('out_parts', [1, 2, 3])
def test_epilogue_operand_format(leaf, act, accumulate, out_parts):
    """the lean epilogue writing the next convolution's operand format: bf16 expansion in 1..3 parts, or e4m3 from e4m3 operands"""
    case = CASE[leaf]
    fp8 = case[8] == 'fp8'
    if fp8 and out_parts > 1:
        pytest.skip('e4m3 output is one part')
    n, o = case[1], case[3]
    oh, ow = case[5] + 2 * case[7] - case[4] + 1, case[6] + 2 * case[7] - case[4] + 1
    xp, pw = operands(case, seed=4)
    ep = _epi_args(case, 'plane', seed=7)
    kw = dict(act=act, alpha=0.2, gain=math.sqrt(2), clamp=2.0)
    dt = torch.float8_e4m3fn if fp8 else torch.bfloat16
    prev = 0.5 * _randn(n, o, oh, ow, seed=9) if accumulate else torch.zeros(n, o, oh, ow, device=DEV)
    data = cg._plugin.pack_activations(prev, None, o, out_parts, e4m3=fp8)
    prev = data.double().sum(0).permute(0, 3, 1, 2)             # what the buffer holds before the launch
    out = cg.PackedAct(data, o)
    y, plan = run(case, xp, pw, out_packed=out, accumulate=accumulate, **ep, **kw)
    got = out.data.double().sum(0).permute(0, 3, 1, 2)
    want = epilogue_ref(case_ref(case, xp, pw)[:, :o], **ep, **kw) + prev
    if fp8:             # e4m3: 3 mantissa bits, subnormal spacing 2^-9
        assert bool(((got - want).abs() <= want.abs() * 2.0 ** -4 + 2.0 ** -10 + 1e-5).all()), float((got - want).abs().max())
    elif out_parts == 3:
        check(got, want, case[8])
    else:
        check_rounded(got, want, 2.0 ** (-8 if out_parts == 1 else -17), 3.0 if accumulate else 1.0)
    assert plan['epilogue'] == 1
    assert_leaf(plan, leaf)


def test_instance_norm_statistics_of_a_stacked_accumulator():
    case = CASE['slab i9 p2 stk']
    xp, pw = operands(case, seed=11)
    ep = _epi_args(case, 'plane', seed=12)
    with plans() as seen:
        y, mean, rstd = cg.igemm_conv(xp, pw, precision=case[8], out_dtype=torch.float32, act='lrelu', alpha=0.2, gain=math.sqrt(2),
                                      instnorm_eps=1e-5, **ep)
    want = epilogue_ref(case_ref(case, xp, pw)[:, :case[3]], act='lrelu', alpha=0.2, gain=math.sqrt(2), **ep)
    check(y, want, case[8])
    var, mu = torch.var_mean(want, dim=(2, 3), unbiased=False)
    assert rel_l2(mean, mu) < 1e-5 and rel_l2(rstd, (var + 1e-5).rsqrt()) < 1e-5, (rel_l2(mean, mu), rel_l2(rstd, (var + 1e-5).rsqrt()))
    assert seen[0]['stack'] == 1 and seen[0]['stats_rows'] > 0
    assert_leaf(seen[0], 'slab i9 p2 stk')


@pytest.mark.parametrize('kind', ['tanh', 'negative_gain', 'several_samples_per_tile'])
def test_general_epilogue(kind):
    """the non-fast path: an activation the gain cannot be folded into, a negative gain, and tiles of several samples (images under
    128 pixels)"""
    case = CASE['slab i9 p2 stk'] if kind != 'several_samples_per_tile' else ('i3 p2', 7, 64, 48, 3, 5, 6, 1, 'bf16x2', ())
    xp, pw = operands(case, seed=13)
    ep = _epi_args(case, 'per_sample', seed=14)
    kw = dict(act='tanh', gain=1.7) if kind == 'tanh' else dict(act='lrelu', alpha=0.2, gain=-0.8 if kind == 'negative_gain' else 1.3, clamp=0.9)
    y, plan = run(case, xp, pw, out_dtype=torch.float32, **ep, **kw)
    check(y, epilogue_ref(case_ref(case, xp, pw)[:, :case[3]], **ep, **kw), case[8])
    assert plan['fast'] == 0 and plan['stack'] == 0 and (plan['tn'] > 1) == (kind == 'several_samples_per_tile')


@pytest.mark.parametrize('prec', ['bf16x2', 'fp8'])
def test_up2_phases_with_o_not_a_multiple_of_16(prec):
    """the polyphase up = 2 form: GEMM column g = phase * phase_stride + oc with phase_stride = 32 > o = 24 (padding columns between
    the phases), output pixel (2y + py, 2x + px)"""
    n, ic, o, h, w = 2, 64, 24, 13, 11
    parts = cg._PRODUCTS[prec][1]
    wt = _randn(o, ic, 3, 3, seed=15) / math.sqrt(ic * 9)
    f = torch.tensor([1.0, 3.0, 3.0, 1.0], device=DEV)
    f = (f[:, None] * f[None, :]) / 64
    pw = cg.packed_up2(wt, f, True, False, parts, e4m3=prec == 'fp8')
    assert pw.phases == 4 and pw.phase_stride == 32
    x = _randn(n, ic, h, w, seed=16)
    xp = cg.PackedAct(cg._plugin.pack_activations(x, None, pw.c_pad, parts, e4m3=prec == 'fp8'), ic)
    ep = dict(noise=0.3 * _randn(n, 1, 2 * h, 2 * w, seed=17), bias=_randn(o, seed=18))
    with plans() as seen:
        y = cg.igemm_conv(xp, pw, precision=prec, out_dtype=torch.float32, act='lrelu', alpha=0.2, gain=math.sqrt(2), **ep)
    wgt = pw.data if pw.data.dim() == 4 else pw.data[None]
    g = gemm_ref(xp.data, wgt, 3, 3, 1, 1, h, w, parts, pw.wscale)            # [n, o_rows, h, w]
    acc = g[:, :4 * 32].reshape(n, 2, 2, 32, h, w)[:, :, :, :o].permute(0, 3, 4, 1, 5, 2).reshape(n, o, 2 * h, 2 * w)
    check(y, epilogue_ref(acc, act='lrelu', alpha=0.2, gain=math.sqrt(2), **ep), prec)
    assert seen[0]['block_n'] >= 32


@pytest.mark.parametrize('prec', ['bf16x2', 'fp8'])
def test_spade_epilogue(prec):
    """gamma | beta of a SPADE block in one accumulator tile, the normalised input modulated in the epilogue"""
    n, ic, c, h, w = 6, 64 if prec != 'fp8' else 128, 32, 64, 64
    case = ('?', n, ic, 2 * c, 3, h, w, 1, prec, ())
    xp, pw = operands(case, seed=19)
    sx = _randn(n, c, h, w, seed=20)
    smean, srstd = 0.1 * _randn(n, c, seed=21), _randn(n, c, seed=22).abs() + 0.5
    bias = 0.2 * _randn(2 * c, seed=23)
    fp8 = prec == 'fp8'
    out = cg.PackedAct(torch.zeros([1 if fp8 else 3, n, h, w, c], dtype=torch.float8_e4m3fn if fp8 else torch.bfloat16, device=DEV), c)
    with plans() as seen:
        cg.igemm_conv(xp, pw, precision=prec, bias=bias, out_packed=out, spade=(sx, smean, srstd, 1.4))
    acc = case_ref(case, xp, pw)[:, :2 * c] + bias.double()[None, :, None, None]
    v = (sx.double() - smean.double()[:, :, None, None]) * srstd.double()[:, :, None, None] * (1 + acc[:, :c]) + acc[:, c:]
    want = v.clamp_min(0) * 1.4
    got = out.data.double().sum(0).permute(0, 3, 1, 2)
    if fp8:
        assert bool(((got - want).abs() <= want.abs() * 2.0 ** -4 + 2.0 ** -10 + 1e-5).all()), float((got - want).abs().max())
    else:
        check(got, want, prec)
    assert seen[0]['block_n'] == 2 * c


# ---- d. per-sample resident weights ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize('leaf', ['i3 p2 res', 'slab i9 p2', 'f8 i3 res', 'f8 slab inner9'])
def test_per_sample_resident_weights(leaf):
    """style-modulated weights per sample on resident-weight issuers, with fewer than 148 tiles per sample: CTAs change sample in the
    middle of their walk and reload the resident weights.  Styles of alternating sign and growing magnitude make weights left over
    from the previous sample an O(1) error in every sample."""
    case = CASE[leaf]
    n, ic = case[1], case[2]
    assert n >= 6
    xp, pw = operands(case, seed=24)
    sign = torch.tensor([(-1.0) ** i * (i + 1) for i in range(n)], device=DEV)
    scale = sign[:, None] * (_randn(n, ic, seed=25).abs() * 0.5 + 0.5)
    y, plan = run(case, xp, pw, scale=scale, out_dtype=torch.float32)
    if case[8] == 'fp8':
        wdata, wsc = cg._plugin.quantize_weights_e4m3(pw.master.reshape(-1, pw.o_rows, pw.c_pad), scale)
        want = case_ref(case, xp, pw, wgt=wdata, wscale=wsc)
    else:
        parts = cg._PRODUCTS[case[8]][1]
        wdata = cg._plugin.modulate_weights(pw.master, scale, parts).reshape(n, parts, case[4] ** 2, pw.o_rows, pw.c_pad)
        want = case_ref(case, xp, pw, wgt=wdata)
    for i in range(n):
        check(y[i], want[i, :case[3]], case[8])
    assert plan['b_resident'] == 1 and plan['total_tiles'] // n < 148 < plan['total_tiles']
    assert_leaf(plan, leaf)


# ---- e. channel blocks narrower than the packers produce, through the C ABI ------------------------------------------------------

@pytest.mark.parametrize('c_pad,fp8,kb', [(16, False, 16), (32, False, 32), (48, False, 16), (32, True, 32), (64, True, 64), (96, True, 32)])
def test_narrow_channel_blocks(c_pad, fp8, kb):
    """c_pad 16 / 32 / 48 (bf16: K blocks of 16 / 32 channels, 32- and 64-byte swizzle rows) and 32 / 64 / 96 (e4m3)"""
    case = CASE['f8 generic' if fp8 else 'generic']
    _, n, _, o, k, h, w, pad, prec, _ = case
    parts = cg._PRODUCTS[prec][1]
    d = case_desc(case)
    d.c_pad = d.act_pixel_stride = c_pad
    cols = d.o_rows
    dt = torch.float8_e4m3fn if fp8 else torch.bfloat16
    act = cg._split_bf16(_randn(n, h, w, c_pad, seed=26), parts) if not fp8 else _randn(1, n, h, w, c_pad, seed=26).to(dt)
    wgt = _randn(k * k, cols, c_pad, seed=27) / math.sqrt(c_pad * k * k)
    wgt[:, o:] = 0
    wgt = cg._split_bf16(wgt, parts) if not fp8 else (wgt * 64).to(dt)[None]
    wscale = torch.full([cols], 1 / 64, device=DEV) if fp8 else None
    out = torch.empty(n, o, d.conv_h, d.conv_w, device=DEV)
    act, wgt = act.contiguous(), wgt.contiguous()
    d.act, d.wgt, d.out = act.data_ptr(), wgt.data_ptr(), out.data_ptr()
    if fp8:
        d.wscale = wscale.data_ptr()
    with plans() as seen:
        cg._plugin.conv2d_igemm(d, DEV)
    torch.cuda.synchronize()
    check(out, gemm_ref(act, wgt, k, k, pad, pad, d.conv_h, d.conv_w, parts, wscale)[:, :o], prec)
    assert seen[0]['kb'] == kb


# ---- f. the ablation switches compute the same convolution ------------------------------------------------------------------------

@pytest.mark.parametrize('leaf', ['slab i9 p2 stk', 'i3 p2 res', 'f8 slab inner9'])
@pytest.mark.parametrize('switch,field,value', [
    ('PGPP_IGEMM_NO_REUSE', 'reuse', 0), ('PGPP_IGEMM_NO_SLAB2', 'reuse', 1), ('PGPP_IGEMM_NO_RESIDENT', 'b_resident', 0),
    ('PGPP_IGEMM_NO_STACK', 'stack', 0), ('PGPP_IGEMM_NO_LEAN_EPILOGUE', 'epilogue', 0)])
def test_switch_equivalence(leaf, switch, field, value):
    case = CASE[leaf]
    fp8 = case[8] == 'fp8'
    xp, pw = operands(case, seed=28)
    n, o = case[1], case[3]
    oh, ow = case[5] + 2 * case[7] - case[4] + 1, case[6] + 2 * case[7] - case[4] + 1
    want = epilogue_ref(case_ref(case, xp, pw)[:, :o], act='lrelu', alpha=0.2, gain=math.sqrt(2))
    results = []
    for env in ((), (switch,)):
        out = cg.PackedAct(torch.zeros([1 if fp8 else 3, n, oh, ow, o], dtype=torch.float8_e4m3fn if fp8 else torch.bfloat16, device=DEV), o)
        with switches(env), plans() as seen:
            cg.igemm_conv(xp, pw, precision=case[8], out_packed=out, act='lrelu', alpha=0.2, gain=math.sqrt(2))
        got = out.data.double().sum(0).permute(0, 3, 1, 2)
        if fp8:
            assert bool(((got - want).abs() <= want.abs() * 2.0 ** -4 + 2.0 ** -10 + 1e-5).all()), float((got - want).abs().max())
        else:
            check(got, want, case[8])
        results.append((got, seen[0]))
    (g0, p0), (g1, p1) = results
    if _b200():
        if fp8 and field == 'epilogue':
            assert p1['epilogue'] == 1             # e4m3 output has only the lean epilogue
        else:
            assert p1[field] == value, (p0, p1)
        if leaf == 'slab i9 p2 stk':
            assert p0[field] != value, p0          # on this leaf every switch changes the launch


def test_zz_report_worst_rel_l2():
    """largest exact-product rel-L2 of this module per precision (printed with -s)"""
    print('\nexact-product rel-L2, worst per precision on', torch.cuda.get_device_name(0),
          f'({torch.cuda.get_device_properties(0).multi_processor_count} SMs):', {k: f'{v:.2e}' for k, v in sorted(WORST.items())})
