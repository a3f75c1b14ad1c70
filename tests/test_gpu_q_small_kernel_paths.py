"""Every instantiation of the small operand kernels (csrc/conv_pack.cu, fir_packed.cu, conv_thin.cu, reduce.cu) against a float64 CPU
reference.  The cases come from small_kernel_leaves.py; each records the pgpp:: kernels it launched (torch.profiler) and checks the one it
names.  Every case runs twice:

- exact: small integers, dyadic scales / gains / slopes / taps, so that every float32 operation of the kernel is exact and the summation
  order cannot matter - the result must equal the reference bit for bit (a dropped tail element shows however large the tensor);
- random: Gaussian inputs, compared elementwise against a bound derived from the kernel's float32 arithmetic (unit roundoff u = 2^-24
  per operation; an operand-format result adds the truncation of its last bf16 part)."""
import ctypes
import importlib
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch.profiler import ProfilerActivity, profile

import small_kernel_leaves as L
from conftest import load_pkg
from fp8_ref import e4m3
from helpers import rel_l2
from oracle import ref_ops

pytestmark = pytest.mark.gpu
load_pkg()
custom_ops = importlib.import_module('pgpp_b200.torch_utils.custom_ops')
cg = importlib.import_module('pgpp_b200.torch_utils.ops.conv2d_gradfix')
nets = importlib.import_module('pgpp_b200.training.networks')
DEV = 'cuda:0'
U = 2.0 ** -24
ACT = {'linear': 1, 'relu': 2, 'lrelu': 3}
TORCH_DTYPE = {L.F32: torch.float32, L.F16: torch.float16, L.BF16: torch.bfloat16, L.F64: torch.float64}
# relative error of the sum of p bf16 parts (each part rounds the remainder of the previous ones to nearest, 8 significand bits: at most
# 2^-8 of it), plus float32 roundings of the value itself
SPLIT_TOL = {1: 2.0 ** -8 + 2.0 ** -22, 2: 2.0 ** -16 + 2.0 ** -22, 3: 2.0 ** -22}
WORST = {}          # family -> (largest error / bound of a random case, the error itself)


@pytest.fixture(scope='module', autouse=True)
def _report():
    yield
    print('\nrandom cases: largest |got - want| / bound per family (the bound is the elementwise float32 error bound)')
    for fam, (ratio, err) in sorted(WORST.items()):
        print(f'  {fam:12s} ratio {ratio:.3e}   |err| {err:.3e}')


def _lib():
    return custom_ops.load_library()


def _plugin():
    return custom_ops.get_plugin('conv2d_plugin')


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)


def _check(status):
    if status != 0:
        raise RuntimeError(_lib().pgpp_last_error().decode())


def launched(fn):
    """run fn under torch.profiler -> (its result, the leaf names of the pgpp:: kernels it launched)"""
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {L.leaf_name(e.key) for e in prof.key_averages() if 'pgpp::' in e.key}
    assert names, 'the profiler recorded no pgpp:: kernel'
    return out, names


def _gen(case, kind):
    return torch.Generator().manual_seed(zlib.crc32((L.case_id(case) + kind).encode()))


def _ints(g, shape, lo, hi):
    return torch.randint(lo, hi + 1, tuple(shape), generator=g).double()


def _dyadic(g, shape, values=(-2.0, -1.0, -0.5, 0.5, 1.0, 2.0)):
    v = torch.tensor(values, dtype=torch.float64)
    return v[torch.randint(0, len(values), tuple(shape), generator=g)]


def split_bf16(v, parts):
    """the kernels' operand format: part p = bf16(v - earlier parts), round to nearest even, in float32"""
    v = v.to(torch.float32)
    out = []
    for _ in range(parts):
        q = v.to(torch.bfloat16)
        out.append(q)
        v = v - q.float()
    return torch.stack(out)


def assert_exact_premise(want):
    """the exact cases rely on a reference that float32 represents exactly"""
    assert torch.equal(want.float().double(), want), 'exact case whose reference is not a float32 value'


def expect_exact(got, want):
    got = got.cpu()
    assert got.dtype == want.dtype and got.shape == want.shape, (got.dtype, want.dtype, got.shape, want.shape)
    if not torch.equal(got, want):
        bad = (got.double() != want.double()).nonzero()
        raise AssertionError(f'{len(bad)} elements differ, first at {bad[0].tolist()}: got {got[tuple(bad[0])]}, want {want[tuple(bad[0])]}')


def expect_close(family, got, want, bound):
    """|got - want| <= bound elementwise (all float64 CPU tensors); the largest ratio is kept for the report"""
    got = got.detach().double().cpu()
    assert got.shape == want.shape, (got.shape, want.shape)
    assert torch.isfinite(got).all()
    err = (got - want).abs()
    ratio = float((err / bound.clamp_min(1e-300)).max())
    prev = WORST.get(family, (0.0, 0.0))
    if ratio > prev[0]:
        WORST[family] = (ratio, float(err.max()))
    assert ratio <= 1.0, (family, ratio, float(err.max()))


def check_packed(family, kind, got_parts, want, extra_bound=None):
    """an operand-format result [parts, ...] (bf16) against the float64 reference value `want` of the same shape without the part axis"""
    parts = got_parts.shape[0]
    if kind == 'exact':
        assert_exact_premise(want)
        expect_exact(got_parts, split_bf16(want, parts))
    else:
        bound = SPLIT_TOL[parts] * want.abs() + (0 if extra_bound is None else extra_bound)
        expect_close(family, got_parts.double().sum(0), want, bound.clamp_min(1e-30))


def apply_act(v, act, alpha, gain, clamp):
    if act == 'relu':
        v = v.clamp_min(0)
    elif act == 'lrelu':
        v = torch.where(v > 0, v, v * alpha)
    v = v * gain
    return v.clamp(-clamp, clamp) if clamp >= 0 else v


def act_bound(bound, act, alpha, gain):
    """a bound on the error before bias_act-style epilogue -> after it (act is 1-Lipschitz up to alpha, clamp does not increase it)"""
    return bound * abs(gain) * (max(1.0, alpha) if act == 'lrelu' else 1.0)


def c_i64x4(*v):
    return custom_ops.c_i64x4(*v)


def _ids(cases):
    return [L.case_id(c) for c in cases]


KINDS = ['exact', 'random']


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_pack_activations / _slice / _f16 / _e4m3

def _source(g, kind, dtype, shape, view):
    """-> (device tensor laid out as `view`, its values as a float64 CPU tensor)"""
    n, c, h, w = shape
    td = TORCH_DTYPE[dtype]
    if kind == 'exact':
        lim = 250 if dtype == L.BF16 else 2000              # exactly representable in the source dtype
        vals = _ints(g, shape, -lim, lim).to(td)
    else:
        vals = torch.randn(shape, generator=g, dtype=torch.float64).to(td)
    if view == 'contig':
        x = vals.to(DEV)
    elif view == 'pitch':
        pitch = w + 4 if w % 4 == 0 else -(-w // 4) * 4
        big = torch.full((n, c, h, pitch), 3.0, dtype=td, device=DEV)
        big[..., :w] = vals.to(DEV)
        x = big[..., :w]
    elif view == 'misaligned':
        x = torch.empty(n * c * h * w + 1, dtype=td, device=DEV)[1:].view(n, c, h, w)
        x.copy_(vals.to(DEV))
    elif view == 'sn_odd':
        store = torch.empty(n * (c * h * w + 1), dtype=td, device=DEV)
        x = store.as_strided((n, c, h, w), (c * h * w + 1, h * w, w, 1))
        x.copy_(vals.to(DEV))
    elif view == 'cl':
        x = vals.to(DEV).contiguous(memory_format=torch.channels_last)
    elif view == 'step2':
        big = torch.zeros((n, c, h, 2 * w), dtype=td, device=DEV)
        big[..., ::2] = vals.to(DEV)
        x = big[..., ::2]
    else:
        raise ValueError(view)
    return x, vals.double()


SENTINEL = 7.0


def _pack_call(x, scale, mode, c_pad, c_total, c_off):
    n, c, h, w = x.shape
    dt = {'e4m3': torch.float8_e4m3fn, 'f16': torch.float16}.get(mode, torch.bfloat16)
    parts = mode if isinstance(mode, int) else 1
    dst = torch.full((parts, n, h, w, c_total), SENTINEL, device=DEV).to(dt)
    lib = _lib()
    args = (ctypes.c_void_p(x.data_ptr()), c_i64x4(*x.shape), c_i64x4(*x.stride()), custom_ops.dtype_code(x.dtype),
            None if scale is None else ctypes.c_void_p(scale.data_ptr()), ctypes.c_void_p(dst.data_ptr()))
    if mode == 'e4m3':
        _check(lib.pgpp_pack_activations_e4m3(*args, c_pad, c_total, c_off, _stream()))
    elif mode == 'f16':
        _check(lib.pgpp_pack_activations_f16(*args, c_pad, c_total, c_off, _stream()))
    else:
        _check(lib.pgpp_pack_activations_slice(*args, c_pad, c_total, c_off, parts, _stream()))
    return dst


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.PACK_CASES, ids=_ids(L.PACK_CASES))
def test_pack_activations(case, kind):
    leaf, dtype, shape, view, mode, c_slice = case
    g = _gen(case, kind)
    n, c, h, w = shape
    x, vals = _source(g, kind, dtype, shape, view)
    c_pad = -(-c // 16) * 16
    c_total, c_off = c_slice if c_slice else (c_pad, 0)
    s = _dyadic(g, (n, c)) if kind == 'exact' else torch.randn(n, c, generator=g, dtype=torch.float64).float().double()
    for scale in (None, s):
        sc = None if scale is None else scale.float().to(DEV)
        dst, names = launched(lambda: _pack_call(x, sc, mode, c_pad, c_total, c_off))
        assert leaf in names, names
        dst = dst.cpu()
        outside = torch.cat([dst[..., :c_off], dst[..., c_off + c_pad:]], -1).float()
        assert torch.all(outside == SENTINEL), 'channels outside the destination slice were written'
        assert torch.all(dst[..., c_off + c:c_off + c_pad].float() == 0), 'padding channels are not zero'
        got = dst[..., c_off:c_off + c]
        v32 = vals.float() if scale is None else vals.float() * scale.float()[:, :, None, None]     # the kernel's float32 product
        v32 = v32.permute(0, 2, 3, 1)
        if mode == 'e4m3':
            expect_exact(got[0], e4m3(v32))
        elif mode == 'f16':
            expect_exact(got[0], v32.half())
        else:
            want = (vals if scale is None else vals * scale[:, :, None, None]).permute(0, 2, 3, 1)
            if kind == 'random':
                expect_exact(got[0], v32.to(torch.bfloat16))                          # the first part rounds the float32 product
            check_packed('pack', kind, got, want)


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_pack_act_gradient

@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.ACT_GRAD_CASES, ids=_ids(L.ACT_GRAD_CASES))
def test_pack_act_gradient(case, kind):
    leaf, dtype, shape, act, alpha, gain, clamp, mode = case
    g = _gen(case, kind)
    n, c, h, w = shape
    td = TORCH_DTYPE[dtype]
    if kind == 'exact':
        dy = _ints(g, shape, -8, 8)
        y = _ints(g, shape, -4, 4)                  # +-3 = +-clamp: the clamp passes the gradient strictly inside
    else:
        dy = torch.randn(shape, generator=g, dtype=torch.float64)
        y = torch.randn(shape, generator=g, dtype=torch.float64) * 2.5
        y.view(-1)[::13] = 3.0
        y.view(-1)[5::13] = -3.0
        y.view(-1)[7::13] = 0.0
    dy, y = dy.to(td), y.to(td)
    c_pad = -(-c // 16) * 16
    f16 = mode == 'f16'
    parts = 1 if f16 else mode
    (out, sums), names = launched(lambda: _plugin().pack_act_gradient(dy.to(DEV), y.to(DEV), ACT[act], alpha, gain, clamp, c_pad, parts,
                                                                      f16=f16, want_sums=True))
    assert leaf in names, names
    dyd, yd = dy.double(), y.double()
    slope = {'linear': 1.0, 'relu': 0.0, 'lrelu': alpha}[act]
    pos = (yd > 0) if gain > 0 else (yd < 0)
    r = torch.where(pos, dyd, dyd * slope) * gain
    if clamp >= 0:
        r = torch.where((yd > -clamp) & (yd < clamp), r, torch.zeros_like(r))
    want = r.permute(0, 2, 3, 1)
    got = out.cpu()[..., :c]
    assert torch.all(out.cpu()[..., c:].float() == 0)
    if kind == 'exact':
        assert_exact_premise(r)
        assert torch.equal(r.to(td).double(), r), 'exact case not representable in the tensor dtype'
        if f16:
            expect_exact(got[0], want.half())
        else:
            expect_exact(got, split_bf16(want, parts))
        expect_exact(sums.cpu().sum(-1).double(), r.sum((2, 3)))
    else:
        t_tol = {torch.float32: 2 * U, torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7}[td]     # two roundings, then through T
        got_v = got[0].double() if f16 else got.double().sum(0)
        expect_close('act_grad', got_v, want, (max(t_tol, 0 if f16 else SPLIT_TOL[parts]) * want.abs() + 1e-30))
        rt = r.float().to(td).double()                                   # what the kernel sums: the value rounded through T
        expect_close('act_grad', sums.cpu().sum(-1), rt.sum((2, 3)), (h * w + 8) * U * rt.abs().sum((2, 3)) + 1e-30)


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_pack_im2col

@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.IM2COL_CASES, ids=_ids(L.IM2COL_CASES))
def test_pack_im2col(case, kind):
    """bit-exact for both kinds: the value is staged in shared memory, so the split is the float32 one of the emulation"""
    leaf, dtype, shape, kw, r, pad_x, pad_y, scaled, parts = case
    g = _gen(case, kind)
    n, c, h, w = shape
    td = TORCH_DTYPE[dtype]
    vals = (_ints(g, shape, -250, 250) if kind == 'exact' else torch.randn(shape, generator=g, dtype=torch.float64)).to(td)
    s = (_dyadic(g, (n, c)) if kind == 'exact' else torch.randn(n, c, generator=g, dtype=torch.float64)).float()
    out, names = launched(lambda: _plugin().pack_im2col(vals.to(DEV), s.to(DEV) if scaled else None, kw, r, pad_x, pad_y, parts))
    assert leaf in names, names
    xs = vals.float() * s[:, :, None, None] if scaled else vals.float()
    xp = F.pad(xs, [pad_x, kw, pad_y, r])
    packed = torch.zeros(n, h + pad_y, w, 64, dtype=torch.float32)
    for ry in range(r):
        for kx in range(kw):
            ch0 = (ry * kw + kx) * c
            packed[..., ch0:ch0 + c] = xp[:, :, ry:ry + h + pad_y, kx:kx + w].permute(0, 2, 3, 1)
    expect_exact(out, split_bf16(packed, parts))


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_spade_modulate_pack, pgpp_mix_pack

@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.SPADE_CASES, ids=_ids(L.SPADE_CASES))
def test_spade_modulate_pack(case, kind):
    leaf, shape, c_pad, parts, pre_gain, gb_pad, x_offset = case
    g = _gen(case, kind)
    n, c, h, w = shape
    if kind == 'exact':
        x, gm, bt = _ints(g, shape, -8, 8), _ints(g, shape, -3, 3), _ints(g, shape, -4, 4)
        mean, rstd = _ints(g, (n, c), -2, 2), _dyadic(g, (n, c), (0.25, 0.5, 1.0, 2.0))
    else:
        x, gm, bt = (torch.randn(shape, generator=g, dtype=torch.float64) for _ in range(3))
        mean, rstd = torch.randn(n, c, generator=g, dtype=torch.float64), torch.rand(n, c, generator=g, dtype=torch.float64) + 0.5
    x, gm, bt, mean, rstd = (t.float() for t in (x, gm, bt, mean, rstd))
    xd = torch.empty(n * c * h * w + x_offset, device=DEV)[x_offset:].view(shape)
    xd.copy_(x.to(DEV))
    sn = c * h * w + gb_pad
    gd, bd = (torch.zeros(n * sn, device=DEV).as_strided(shape, (sn, h * w, w, 1)) for _ in range(2))
    gd.copy_(gm.to(DEV)); bd.copy_(bt.to(DEV))
    md, rd = mean.to(DEV), rstd.to(DEV)
    out = torch.full((parts, n, h, w, c_pad), SENTINEL, device=DEV).to(torch.bfloat16)
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    _, names = launched(lambda: _check(_lib().pgpp_spade_modulate_pack(P(xd), P(md), P(rd), P(gd), P(bd), sn, P(out), n, c, h, w, c_pad, parts,
                                                                       float(pre_gain), _stream())))
    assert leaf in names, names
    xd64, m64, r64 = x.double(), mean.double()[:, :, None, None], rstd.double()[:, :, None, None]
    t = (xd64 - m64) * r64
    v = t * (1 + gm.double()) + bt.double()
    if pre_gain > 0:
        v = v.clamp_min(0) * pre_gain
    got = out.cpu()
    assert torch.all(got[..., c:].float() == 0)
    bound = None
    if kind == 'random':    # x - mean, * rstd, 1 + gamma, fma: 4 roundings of terms of size |t (1 + gamma)| + |beta|
        bound = 4 * U * ((t.abs() * (1 + gm.double()).abs()) + bt.double().abs() + (xd64.abs() + m64.abs()) * r64 * (1 + gm.double()).abs())
        bound = (bound * max(1.0, pre_gain)).permute(0, 2, 3, 1)
    check_packed('spade', kind, got[..., :c], v.permute(0, 2, 3, 1), bound)


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.MIX_CASES, ids=_ids(L.MIX_CASES))
def test_mix_pack(case, kind):
    leaf, shape, c_pad, parts, n_terms, misaligned = case
    g = _gen(case, kind)
    n, c, h, w = shape
    draw = (lambda s: _ints(g, s, -8, 8)) if kind == 'exact' else (lambda s: torch.randn(s, generator=g, dtype=torch.float64))
    terms = [(draw(shape).float(), draw((n, c)).float(), draw((n, h, w)).float(), draw((n, h, w)).float()) for _ in range(n_terms)]

    def dev(t):
        if not misaligned:
            return t.to(DEV)
        d = torch.empty(t.numel() + 1, device=DEV)[1:].view(t.shape)
        d.copy_(t.to(DEV))
        return d
    dterms = [tuple(dev(t) for t in term) for term in terms]
    out, names = launched(lambda: _plugin().mix_pack(dterms, c_pad, parts))
    assert leaf in names, names
    want = torch.zeros(shape, dtype=torch.float64)
    mag = torch.zeros(shape, dtype=torch.float64)
    for x, m, a, b in terms:
        xa, mb = x.double() * a.double()[:, None], m.double()[:, :, None, None] * b.double()[:, None]
        want += xa + mb
        mag += xa.abs() + mb.abs()
    got = out.cpu()
    assert torch.all(got[..., c:].float() == 0)
    check_packed('mix', kind, got[..., :c], want.permute(0, 2, 3, 1), (2 * n_terms + 1) * U * mag.permute(0, 2, 3, 1))


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_conv2d_direct

@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.DIRECT_CASES, ids=_ids(L.DIRECT_CASES))
def test_conv2d_direct(case, kind):
    leaf, n, c, h, w, o, kh, kw, act, clamp, packed = case
    g = _gen(case, kind)
    wscale, alpha, gain = 0.5, 0.25, 0.5
    if kind == 'exact':
        x, wt, b = _ints(g, (n, c, h, w), -4, 4), _ints(g, (o, c, kh, kw), -3, 3), _ints(g, (o,), -4, 4)
    else:
        x, wt, b = (torch.randn(s, generator=g, dtype=torch.float64) for s in ((n, c, h, w), (o, c, kh, kw), (o,)))
    x, wt, b = x.float(), wt.float(), b.float()
    buf = None
    if packed:
        parts, c_total, c_off = packed
        buf = torch.full((parts, n, h, w, c_total), SENTINEL, device=DEV).to(torch.bfloat16)
    run = lambda: _plugin().conv2d_direct(x.to(DEV), wt.to(DEV), b.to(DEV), wscale, ACT[act], alpha, gain, clamp,
                                          out_packed_data=buf, c_off=packed[2] if packed else 0)
    out, names = launched(run)
    assert leaf in names, names
    ws = (wt * wscale).double()                                         # the kernel stages w * wscale in float32
    pre = F.conv2d(x.double(), ws, b.double(), padding=(kh // 2, kw // 2))
    want = apply_act(pre, act, alpha, gain, clamp)
    bound = None
    if kind == 'random':
        bound = act_bound((c * kh * kw + 2) * U * (F.conv2d(x.double().abs(), ws.abs(), padding=(kh // 2, kw // 2)) + b.double().abs()[:, None, None]),
                          act, alpha, gain) + U * want.abs()
    if packed is None:
        if kind == 'exact':
            assert_exact_premise(want)
            expect_exact(out.cpu(), want.float())
        else:
            expect_close('direct', out, want, bound)
        return
    parts, c_total, c_off = packed
    got = buf.cpu()
    outside = torch.cat([got[..., :c_off], got[..., c_off + o:]], -1).float()
    assert torch.all(outside == SENTINEL), 'channels outside the destination slice were written'
    check_packed('direct', kind, got[..., c_off:c_off + o], want.permute(0, 2, 3, 1), None if bound is None else bound.permute(0, 2, 3, 1))


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_modconv_demod_coefs, pgpp_modulate_weights

@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.DEMOD_CASES, ids=_ids(L.DEMOD_CASES))
def test_demod_coefs(case, kind):
    """the sums are exact in the exact case; rsqrtf itself is within 2 ulp (CUDA C Programming Guide, mathematical functions)"""
    leaf, n, o, i, kh, kw = case
    g = _gen(case, kind)
    if kind == 'exact':
        wt, s, eps = _ints(g, (o, i, kh, kw), -3, 3), _ints(g, (n, i), -2, 2), 1.0
    else:
        wt, s, eps = torch.randn(o, i, kh, kw, generator=g, dtype=torch.float64), torch.randn(n, i, generator=g, dtype=torch.float64), 1e-8
    wt, s = wt.float(), s.float()
    d, names = launched(lambda: _plugin().demod_coefs(wt.to(DEV), s.to(DEV), eps))
    assert leaf in names, names
    ssum = torch.einsum('oi,ni->no', wt.double().square().sum((2, 3)), s.double().square())
    want = (ssum + eps).rsqrt()
    if kind == 'exact':
        assert_exact_premise(ssum)
        expect_close('demod_exact', d, want, 2.0 ** -22 * want)
    else:
        expect_close('demod', d, want, (2.0 ** -22 + (i * kh * kw + i + 64) * U / 2) * want)


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.MODW_CASES, ids=_ids(L.MODW_CASES))
def test_modulate_weights(case, kind):
    leaf, n, rows, c_pad, c_in, parts = case
    g = _gen(case, kind)
    if kind == 'exact':
        master, s = _ints(g, (rows, c_pad), -2000, 2000), _dyadic(g, (n, c_in))
    else:
        master, s = torch.randn(rows, c_pad, generator=g, dtype=torch.float64), torch.randn(n, c_in, generator=g, dtype=torch.float64)
    master, s = master.float(), s.float()
    out, names = launched(lambda: _plugin().modulate_weights(master.to(DEV), s.to(DEV), parts))
    assert leaf in names, names
    got = out.cpu()                                                     # [n, parts, rows, c_pad]
    assert torch.all(got[..., c_in:].float() == 0)
    v32 = master[None, :, :c_in] * s[:, None, :]
    if kind == 'random':
        expect_exact(got[:, 0, :, :c_in], v32.to(torch.bfloat16))
    want = master.double()[None, :, :c_in] * s.double()[:, None, :]
    check_packed('modw', kind, got[..., :c_in].transpose(0, 1), want)


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_fir_pack (float32 NCHW -> operand format)

@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.FIR_PACK_CASES, ids=_ids(L.FIR_PACK_CASES))
def test_fir_pack(case, kind):
    leaf, shape, taps, fh, fw, pad, flip, gain, parts = case
    g = _gen(case, kind)
    n, c, h, w = shape
    x = (_ints(g, shape, -8, 8) if kind == 'exact' else torch.randn(shape, generator=g, dtype=torch.float64)).float()
    c_pad = -(-c // 16) * 16
    out, names = launched(lambda: _plugin().fir_pack(x.to(DEV), taps, fw, fh, *pad, flip, gain, c_pad, parts))
    assert leaf in names, names
    f = torch.tensor(taps, dtype=torch.float32).reshape(fh, fw)
    want = ref_ops.upfirdn2d(x.double(), f, padding=list(pad), flip_filter=flip, gain=gain)
    bound = (fh * fw + 1) * U * ref_ops.upfirdn2d(x.double().abs(), f.abs(), padding=list(pad), flip_filter=flip, gain=abs(gain))
    got = out.cpu()
    assert torch.all(got[..., c:].float() == 0)
    check_packed('fir_pack', kind, got[..., :c], want.permute(0, 2, 3, 1), bound.permute(0, 2, 3, 1))


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_fir_packed / pgpp_fir_packed_act (operand format -> operand format or float32 NCHW)

_NS4X4 = [1, 2, 0, -1, 3, 1, 2, 0, 0, -2, 1, 3, 2, 0, -1, 1]
_NS3X2 = [1, -2, 3, 2, 0, 1]


def _fir_filter(name, kind):
    """-> (taps row-major, fh, fw)"""
    if name == 'sep121':
        return np.outer([1, 2, 1], [1, 2, 1]).ravel().tolist(), 3, 3
    if name == 'sep1331':       # the production blur; its column ratios to the pivot (1/3) are not dyadic, so the exact case uses [1,2,2,1]
        k = [1, 3, 3, 1] if kind == 'random' else [1, 2, 2, 1]
        return np.outer(k, k).ravel().tolist(), 4, 4
    if name == 'ns4x4':
        return _NS4X4, 4, 4
    if name == 'ns3x2':
        return _NS3X2, 3, 2
    return None, 1, 1


def _packed_source(g, kind, parts, n, h, w, c, ct, c_off):
    """bf16 [parts, n, h, w, ct] with channels [c_off, c_off + c) the operand; other channels hold a large value that must not be read.
    Exact: the parts are integers, 1/64 and 1/1024 multiples, so that their float32 sum and every filtered sum stays exact."""
    src = torch.full((parts, n, h, w, ct), 1e4, dtype=torch.float64)
    if kind == 'exact':
        scales = [1.0, 2.0 ** -6, 2.0 ** -10]
        for p in range(parts):
            src[p, ..., c_off:c_off + c] = _ints(g, (n, h, w, c), -16 if p == 0 else -31, 16 if p == 0 else 31) * scales[p]
        src = src.to(torch.bfloat16)
    else:
        v = torch.randn(n, h, w, c, generator=g, dtype=torch.float64)
        src = src.to(torch.bfloat16)
        src[..., c_off:c_off + c] = split_bf16(v, parts)
    x = src[..., c_off:c_off + c].double().sum(0).permute(0, 3, 1, 2)        # what the kernel reads: the sum of the parts
    return src, x


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.FIR_PACKED_CASES, ids=_ids(L.FIR_PACKED_CASES))
def test_fir_packed(case, kind):
    leaf, n, c, h, w, in_parts, out_parts, filt, down, pad, flip, gain, epi = case
    g = _gen(case, kind)
    taps, fh, fw = _fir_filter(filt, kind)
    src_off = 8
    src, x = _packed_source(g, kind, in_parts, n, h, w, c, c + 16, src_off)
    src_d = src.to(DEV)
    oh, ow = (h + pad[2] + pad[3] - fh) // down + 1, (w + pad[0] + pad[1] - fw) // down + 1
    f = torch.tensor(taps if taps else [1.0], dtype=torch.float32).reshape(fh, fw)
    want = ref_ops.upfirdn2d(x, f, down=down, padding=list(pad), flip_filter=flip, gain=gain)
    bound = (fh * fw + 1) * U * ref_ops.upfirdn2d(x.abs(), f.abs(), down=down, padding=list(pad), flip_filter=flip, gain=abs(gain))
    dst_c_off = epi['dst_c_off'] if epi else 0
    nchw = epi.get('nchw') if epi else None
    dst = None if nchw else torch.full((out_parts, n, oh, ow, dst_c_off + c + 8), SENTINEL, device=DEV).to(torch.bfloat16)
    if epi is None or filt is None:
        run = lambda: _plugin().fir_packed(src_d, c, src_off, taps, fw, fh, down, *pad, flip, gain, dst=dst, dst_c_off=dst_c_off)
    else:
        act, alpha, act_gain, clamp = epi['act'], epi['alpha'], epi['gain'], epi['clamp']
        if kind == 'exact':
            noise = {'hw': _ints(g, (oh, ow), -4, 4) / 4, 'nhw': _ints(g, (n, oh, ow), -4, 4) / 4, None: None}[epi['noise']]
            bias = _ints(g, (c,), -4, 4) if epi['bias'] else None
        else:
            noise = {'hw': torch.randn(oh, ow, generator=g, dtype=torch.float64), 'nhw': torch.randn(n, oh, ow, generator=g, dtype=torch.float64),
                     None: None}[epi['noise']]
            bias = torch.randn(c, generator=g, dtype=torch.float64) if epi['bias'] else None
        noise = None if noise is None else noise.float()
        bias = None if bias is None else bias.float()
        pre = want + (0 if noise is None else (noise.double() if noise.dim() == 2 else noise.double()[:, None]))
        pre = pre + (0 if bias is None else bias.double()[:, None, None])
        bound = act_bound(bound + 2 * U * (pre.abs() + (0 if bias is None else bias.double().abs()[:, None, None])), act, alpha, act_gain)
        want = apply_act(pre, act, alpha, act_gain, clamp)
        bound = bound + U * want.abs()
        out_nchw = torch.full((n, nchw, oh, ow), SENTINEL, device=DEV) if nchw else None
        nd = None if noise is None else noise.to(DEV)
        bd = None if bias is None else bias.to(DEV)
        P = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        f_host = (ctypes.c_float * len(taps))(*[float(t) for t in taps])
        lib = _lib()

        def run():
            _check(lib.pgpp_fir_packed_act(
                ctypes.c_void_p(src_d.data_ptr() + 2 * src_off), in_parts, src_d[0].numel(), n, h, w, c, c + 16, f_host, fw, fh, *pad,
                int(flip), float(gain), P(nd), oh * ow if (nd is not None and nd.dim() == 3) else 0, P(bd), ACT[act], float(alpha),
                float(act_gain), float(clamp),
                None if dst is None else ctypes.c_void_p(dst.data_ptr() + 2 * dst_c_off), 0 if dst is None else out_parts,
                0 if dst is None else dst[0].numel(), 0 if dst is None else dst.shape[4], P(out_nchw), nchw or c, _stream()))
            return out_nchw
    out, names = launched(run)
    assert leaf in names, names
    if nchw:
        if kind == 'exact':
            assert_exact_premise(want)
            expect_exact(out.cpu(), want[:, :nchw].float())
        else:
            expect_close('fir_packed', out, want[:, :nchw], bound[:, :nchw])
        return
    got = dst.cpu()
    outside = torch.cat([got[..., :dst_c_off], got[..., dst_c_off + c:]], -1).float()
    assert torch.all(outside == SENTINEL), 'channels outside the destination slice were written'
    if filt is None:            # the channel-slice copy moves every part unchanged
        expect_exact(got[..., dst_c_off:dst_c_off + c], src[..., src_off:src_off + c])
        return
    check_packed('fir_packed', kind, got[..., dst_c_off:dst_c_off + c], want.permute(0, 2, 3, 1), bound.permute(0, 2, 3, 1))


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_conv1x1_thin

@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.THIN_CASES, ids=_ids(L.THIN_CASES))
def test_conv1x1_thin(case, kind):
    leaf, n, c, h, w, parts, o1, o2, c_off, accumulate1, act, clamp = case
    g = _gen(case, kind)
    alpha, gain = 0.25, 0.5
    src, x = _packed_source(g, kind, parts, n, h, w, c, c_off + c + 8, c_off)
    if kind == 'exact':
        w1, w2, b1, b2 = _ints(g, (o1, c), -3, 3), _ints(g, (max(o2, 1), c), -3, 3), _ints(g, (o1,), -4, 4), _ints(g, (max(o2, 1),), -4, 4)
        s = _dyadic(g, (n, c), (-2.0, -1.0, 1.0, 2.0))
        init1 = _ints(g, (n, o1, h, w), -4, 4)
    else:
        w1, w2, b1, b2 = (torch.randn(sh, generator=g, dtype=torch.float64) for sh in ((o1, c), (max(o2, 1), c), (o1,), (max(o2, 1),)))
        s = torch.randn(n, c, generator=g, dtype=torch.float64)
        init1 = torch.randn(n, o1, h, w, generator=g, dtype=torch.float64)
    w1, w2, b1, b2, s, init1 = (t.float() for t in (w1, w2, b1, b2, s, init1))
    w2, b2 = w2[:o2], b2[:o2]
    wall = torch.cat([w1, w2]).double()
    ws = (wall.float()[None] * s[:, None, :]).double()                 # the kernel's float32 w * s
    pre = torch.einsum('nchw,noc->nohw', x, ws) + torch.cat([b1, b2]).double()[None, :, None, None]
    if clamp >= 0:      # clamp the largest values only, at a power of two
        clamp = float(2.0 ** np.floor(np.log2(float(apply_act(pre, act, alpha, gain, -1.0).abs().max()))))
    want = apply_act(pre, act, alpha, gain, clamp)
    bound = act_bound((c + 8) * U * (torch.einsum('nchw,noc->nohw', x.abs(), ws.abs()) + torch.cat([b1, b2]).double().abs()[None, :, None, None]),
                      act, alpha, gain) + U * want.abs()
    if accumulate1:
        want[:, :o1] += init1.double()
        bound[:, :o1] += U * want[:, :o1].abs()
    out1 = init1.to(DEV) if accumulate1 else torch.full((n, o1, h, w), SENTINEL, device=DEV)
    out2 = torch.full((n, o2, h, w), SENTINEL, device=DEV) if o2 else None
    src_d = src.to(DEV)
    _, names = launched(lambda: _plugin().conv1x1_thin(src_d, c, c_off, w1.to(DEV), b1.to(DEV), out1, accumulate1,
                                                       w2.to(DEV) if o2 else None, b2.to(DEV) if o2 else None, out2, styles=s.to(DEV),
                                                       act_idx=ACT[act], alpha=alpha, gain=gain, clamp=clamp))
    assert leaf in names, names
    got = torch.cat([out1, out2], 1) if o2 else out1
    if kind == 'exact':
        assert_exact_premise(want)
        expect_exact(got.cpu(), want.float())
    else:
        expect_close('thin', got, want, bound)


def test_conv1x1_thin_refuses_what_it_does_not_cover():
    src = torch.zeros(1, 1, 4, 4, 512, dtype=torch.bfloat16, device=DEV)
    out = lambda o: torch.zeros(1, o, 4, 4, device=DEV)
    w = lambda o, c: torch.zeros(o, c, device=DEV)
    with pytest.raises(RuntimeError, match='at most 8 output channels'):
        _plugin().conv1x1_thin(src, 64, 0, w(4, 64), None, out(4), False, w(5, 64), None, out(5))
    with pytest.raises(RuntimeError, match='c <= 256'):
        _plugin().conv1x1_thin(src, 512, 0, w(5, 512), None, out(5), False)
    _plugin().conv1x1_thin(src, 512, 0, w(4, 512), None, out(4), False)          # 4 outputs at 512 channels are covered


# ---------------------------------------------------------------------------------------------------------------------------------
# pgpp_mul_reduce_hw, pgpp_sum_hw

def _hw2(hw):
    h = int(np.sqrt(hw))
    while hw % h:
        h -= 1
    return h, hw // h


def _device_copy(t, misaligned):
    if not misaligned:
        return t.to(DEV)
    d = torch.empty(t.numel() + 1, dtype=t.dtype, device=DEV)[1:].view(t.shape)
    d.copy_(t.to(DEV))
    return d


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.MUL_REDUCE_CASES, ids=_ids(L.MUL_REDUCE_CASES))
def test_mul_reduce_hw(case, kind):
    leaf, n, c, hw, with_b, sub_kind, with_scale, out_kind, misaligned = case
    g = _gen(case, kind)
    h, w = _hw2(hw)
    draw = (lambda sh: _ints(g, sh, -4, 4)) if kind == 'exact' else (lambda sh: torch.randn(sh, generator=g, dtype=torch.float64))
    a, b = draw((n, c, h, w)).float(), draw((n, c, h, w)).float()
    sub = {'hw': (h, w), 'n1hw': (n, 1, h, w), '11hw': (1, 1, h, w), None: None}[sub_kind]
    sub = None if sub is None else draw(sub).float()
    scale = (_dyadic(g, (n, c)) if kind == 'exact' else torch.randn(n, c, generator=g, dtype=torch.float64)).float()
    ad = _device_copy(a, misaligned)
    bd = b.to(DEV) if with_b else None
    sd = None if sub is None else sub.to(DEV)
    scd = scale.to(DEV) if with_scale else None
    per_sample_sub = sub_kind == 'n1hw' and n > 1
    if out_kind == 'alias':     # grad_x written over grad_xs: out_scaled == a
        r = torch.empty(n, c, device=DEV)
        P = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        run = lambda: (_check(_lib().pgpp_mul_reduce_hw(P(ad), P(bd), P(sd), hw if per_sample_sub else 0, P(scd), P(ad), P(r), n, c, hw,
                                                        _stream())), (r, ad))[1]
    else:
        run = lambda: _plugin().mul_reduce_hw(ad, bd, sub=sd, scale=scd, out_scaled=out_kind == 'new')
    (r, out), names = launched(run)
    assert leaf in names, names
    bb = b.double() if with_b else torch.ones_like(a.double())
    mag = bb.abs()
    if sub is not None:
        sub64 = sub.double().reshape(n if per_sample_sub else 1, 1, h, w)
        bb, mag = bb - sub64, mag + sub64.abs()
    want = (a.double() * bb).sum((2, 3))
    if kind == 'exact':
        assert_exact_premise(want)
        expect_exact(r.cpu(), want.float())
    else:
        G = 256 if hw >= 2048 else 32
        expect_close('mul_reduce', r, want, (hw // G + 12) * U * (a.double().abs() * mag).sum((2, 3)))
    if out_kind:
        expect_exact(out.cpu(), a * scale[:, :, None, None])           # one float32 product: bit-exact for both kinds


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('case', L.SUM_HW_CASES, ids=_ids(L.SUM_HW_CASES))
def test_sum_hw(case, kind):
    leaf, dtype, n, c, hw, misaligned = case
    g = _gen(case, kind)
    h, w = _hw2(hw)
    td = TORCH_DTYPE[dtype]
    a = (_ints(g, (n, c, h, w), -4, 4) if kind == 'exact' else torch.randn(n, c, h, w, generator=g, dtype=torch.float64)).to(td)
    ad = _device_copy(a, misaligned)
    r, names = launched(lambda: _plugin().sum_hw(ad))
    assert leaf in names, names
    want = a.double().sum((2, 3))
    if kind == 'exact':
        expect_exact(r.cpu(), want.float())
    else:
        G = 256 if hw >= 2048 else 32
        expect_close('sum_hw', r, want, (hw // G + 12) * U * a.double().abs().sum((2, 3)))


# ---------------------------------------------------------------------------------------------------------------------------------
# end to end: the training-mode modulated convolution at a production size

def test_fused_modulated_conv_backward_full_size():
    """_FusedModulatedConv2d (64 -> 64, 3x3, 128 x 128, batch 2): output and the x / weight / style / noise gradients against float64
    autograd of the oracle's formulation.  hw = 16384 takes the one-plane-per-CTA reduction (mul_reduce_kernel<256>) for grad_x,
    grad_styles and the demodulation gradient, as every generator layer from 64 x 64 up does in training."""
    old = cg.fp32_precision
    cg.fp32_precision = 'bf16x3'
    try:
        g = torch.Generator().manual_seed(64)
        n, ic, oc, k, h, w = 2, 64, 64, 3, 128, 128
        x0, w0 = torch.randn(n, ic, h, w, generator=g), torch.randn(oc, ic, k, k, generator=g)
        s0, nz0 = torch.randn(n, ic, generator=g) * 0.5 + 1, torch.randn(h, w, generator=g) * 0.1
        probe = torch.randn(n, oc, h, w, generator=g)

        def run(fn, dev, dt):
            x, wt, s, nz = (v.to(dev, dt).requires_grad_(True) for v in (x0, w0, s0, nz0))
            y = fn(x, wt, s, noise=nz, padding=1, demodulate=True, flip_weight=True, fused_modconv=False)
            grads = torch.autograd.grad((y * probe.to(dev, dt)).sum() + 0.1 * y.square().sum(), [x, wt, s, nz])
            return [y] + list(grads)

        want = run(ref_ops.modulated_conv2d, 'cpu', torch.float64)
        got, names = launched(lambda: run(nets.modulated_conv2d, DEV, torch.float32))
        assert 'mul_reduce_kernel<256>' in names, names
        for a, r, name in zip(got, want, ['y', 'grad_x', 'grad_w', 'grad_s', 'grad_noise']):
            assert rel_l2(a, r) < 1e-4, (name, rel_l2(a, r))     # 2.5x the bf16x3 per-layer tolerance of test_gpu_c_conv
    finally:
        cg.fp32_precision = old
