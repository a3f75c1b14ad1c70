"""CPU tests of the e4m3 emulation the fp8 GPU tests compare the kernels against (tests/fp8_ref.py)."""
import torch

from fp8_ref import E4M3_MAX, conv_from_taps, dequant_weights, e4m3, quantize_weights


def _bytes(t):
    return e4m3(torch.tensor(t, dtype=torch.float32)).view(torch.uint8).tolist()


def test_round_to_nearest_even():
    # [1, 2) has a step of 1/8: the midpoints round to the even mantissa
    got = e4m3(torch.tensor([1.0625, 1.1875, 1.3125, 1.07, -1.0625])).to(torch.float32).tolist()
    assert got == [1.0, 1.25, 1.25, 1.125, -1.0]
    # [256, 448]: step 32
    assert e4m3(torch.tensor([272.0, 304.0, 447.0])).to(torch.float32).tolist() == [256.0, 320.0, 448.0]


def test_subnormals_and_zero():
    m = 2.0 ** -9                                           # smallest subnormal
    got = e4m3(torch.tensor([m, 2 * m, 7 * m, 0.5 * m, 0.75 * m, 1.5 * m, 2.0 ** -6])).to(torch.float32).tolist()
    assert got == [m, 2 * m, 7 * m, 0.0, m, 2 * m, 2.0 ** -6]   # 0.5 m ties to 0 (even), 1.5 m ties to 2 m
    assert _bytes([m, 0.0, -0.0]) == [0x01, 0x00, 0x80]     # +-0 keep their sign bit


def test_saturation():
    got = e4m3(torch.tensor([448.0, 460.0, 464.0, 1e6, -500.0, float('inf'), -float('inf')])).to(torch.float32).tolist()
    assert got == [448.0, 448.0, 448.0, 448.0, -448.0, 448.0, -448.0]
    assert _bytes([448.0, -448.0]) == [0x7E, 0xFE]
    assert torch.isnan(e4m3(torch.tensor([float('nan')])).to(torch.float32)).all()


def test_weight_quantization_scales():
    g = torch.Generator().manual_seed(5)
    master = torch.randn(9, 32, 64, generator=g)
    master[:, 3] = 0.0                                      # an all-zero column: scale 0, bytes 0
    master[:, 5, 7] = 0.0
    master[4, 5, 7] = -3.5                                  # the column's absmax maps to -448
    q, s = quantize_weights(master)
    assert q.shape == (1, 9, 32, 64) and s.shape == (1, 32)
    assert float(s[0, 3]) == 0.0 and (q[0, :, 3].view(torch.uint8) == 0).all()
    assert float(s[0, 5]) == torch.tensor(3.5) / E4M3_MAX
    assert float(q[0, 4, 5, 7].to(torch.float32)) == -448.0
    amax_code = q.to(torch.float32).abs().amax(dim=(1, 3))
    assert bool(((amax_code == 448.0) | (s == 0)).all())
    # per-sample weights: the styles multiply before the absmax; channels beyond c_in are zero
    styles = torch.rand(2, 40, generator=g) + 0.5
    q2, s2 = quantize_weights(master, styles)
    assert q2.shape == (2, 9, 32, 64) and (q2[:, :, :, 40:].view(torch.uint8) == 0).all()
    v = master[None, :, :, :40] * styles[:, None, None, :]
    assert torch.equal(s2, v.abs().amax(dim=(1, 3)) / E4M3_MAX)


def test_dequantized_conv_matches_quantized_operands():
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 16, 8, 8, generator=g)
    w = torch.randn(8, 16, 3, 3, generator=g)
    taps = w.permute(2, 3, 0, 1).reshape(9, 8, 16)          # packed layout: [tap][o][c]
    q, s = quantize_weights(taps)
    wd = dequant_weights(q[0], s[0])
    got = conv_from_taps(e4m3(x).to(torch.float64), wd, 8, 3, 3, padding=(1, 1))
    want = torch.nn.functional.conv2d(x.double(), w.double(), padding=1)
    err = float((got - want).norm() / want.norm())
    assert 5e-3 < err < 8e-2, err                           # e4m3 operands: a few percent per layer
