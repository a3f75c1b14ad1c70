"""Reference emulation of the fp8 (e4m3) operand format (fp32_precision = 'fp8'), shared by the fp8 tests.

torch's float32 -> float8_e4m3fn cast rounds to nearest even but turns values beyond the format (>= 464 in magnitude) into NaN, while
the kernels convert with satfinite (cvt.rn.satfinite.e4m3x2.f32: +-448).  Clamping to +-448 first makes the cast match the kernels."""
import torch
import torch.nn.functional as F

E4M3_MAX = 448.0


def e4m3(x):
    """float tensor -> float8_e4m3fn, round to nearest even, saturating at +-448 (NaN stays NaN)"""
    return x.to(torch.float32).clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn)


def quantize_weights(master, styles=None):
    """What pgpp_quantize_weights_e4m3 writes: master float32 [taps, o_rows, c_pad] (times styles [N, c_in] per sample) ->
    (bytes float8_e4m3fn [N, taps, o_rows, c_pad], column scales float32 [N, o_rows]), scale = absmax / 448 per (sample, column)."""
    m = master.to(torch.float32)
    if styles is None:
        v = m[None]
    else:
        n, c_in = styles.shape
        v = torch.zeros([n, *m.shape], dtype=torch.float32, device=m.device)     # +0 beyond c_in, as the kernel writes
        v[..., :c_in] = m[None, :, :, :c_in] * styles.to(torch.float32)[:, None, None, :]
    amax = v.abs().amax(dim=(1, 3))                         # [N, o_rows]
    scale = amax / torch.full_like(amax, E4M3_MAX)         # a true division (torch may multiply by the reciprocal of a scalar divisor)
    safe = torch.where(scale > 0, scale, torch.ones_like(scale))
    q = torch.where(scale[:, None, :, None] > 0, v / safe[:, None, :, None], torch.zeros_like(v))
    return e4m3(q), scale


def dequant_weights(data, wscale):
    """e4m3 weight rows [taps, o_rows, c_pad] with column scales [o_rows] -> float64 [taps, o_rows, c_pad]"""
    return data.to(torch.float64) * wscale.to(torch.float64)[None, :, None]


def conv_from_taps(x, w_taps, o, kh, kw, stride=1, padding=(0, 0)):
    """float64 correlation of x [N, C, H, W] with the tap-major weight rows w_taps [kh * kw, >= o, >= C] (the packed operand layout)"""
    c = x.shape[1]
    wk = w_taps[:, :o, :c].reshape(kh, kw, o, c).permute(2, 3, 0, 1).contiguous()
    return F.conv2d(x.to(torch.float64), wk, stride=stride, padding=padding)
