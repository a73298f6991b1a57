"""CPU checks of the FP8 inference path's arithmetic: the oracle's e4m3 rounding against a hand table, and the weight
quantisation and epilogue-constant formulas (iswm_b200/quant.py, oracle/torch_model_f8.py) against a numpy restatement."""
import numpy as np
import torch

from iswm_b200 import quant
from oracle import torch_model_f8 as TF8

# (input, e4m3 value): ties to even, saturation to 448 (torch's own cast gives NaN from 480 on), subnormals (2^-9 steps)
E4M3_CASES = [
    (0.0, 0.0), (1.0, 1.0), (-1.0, -1.0),
    (1.0625, 1.0),            # halfway 1 / 1.125: even mantissa 0
    (1.1875, 1.25),           # halfway 1.125 / 1.25: even mantissa 2
    (3.3, 3.25), (-0.3, -0.3125),
    (240.0, 240.0), (248.0, 256.0),   # halfway 240 / 256 (mantissa 7 / exponent up): even
    (416.0, 416.0), (440.0, 448.0), (448.0, 448.0),
    (449.0, 448.0), (464.0, 448.0), (480.0, 448.0), (1e6, 448.0), (-1e6, -448.0), (float("inf"), 448.0),
    (2.0 ** -6, 2.0 ** -6),   # smallest normal
    (2.0 ** -9, 2.0 ** -9),   # smallest subnormal
    (2.0 ** -10, 0.0),        # halfway 0 / 2^-9: even (0)
    (3 * 2.0 ** -10, 2.0 ** -8),   # halfway 2^-9 / 2^-8: even mantissa 2
    (5 * 2.0 ** -10, 2.0 ** -8),   # halfway 2^-8 / 3 * 2^-9: even mantissa 2
    (0.7 * 2.0 ** -9, 2.0 ** -9), (0.4 * 2.0 ** -9, 0.0),
]


def test_e4m3_rounding_hand_table():
    x = torch.tensor([a for a, _ in E4M3_CASES], dtype=torch.float32)
    got = TF8.e4m3(x)
    want = torch.tensor([b for _, b in E4M3_CASES], dtype=torch.float32)
    assert torch.equal(got, want), [(a, float(g)) for (a, _), g in zip(E4M3_CASES, got) if float(g) != _]
    assert not torch.isnan(got).any()


def _np_e4m3(v: np.ndarray) -> np.ndarray:
    """Independent e4m3 rounding: nearest of the 253 finite non-negative e4m3 values (ties to the even code), sign kept."""
    codes = np.arange(0, 127, dtype=np.int64)                     # 0x00 .. 0x7e (0x7f is NaN)
    e, m = codes >> 3, codes & 7
    vals = np.where(e == 0, m * 2.0 ** -9, (1 + m / 8.0) * 2.0 ** (e - 7))
    shape, v = v.shape, v.reshape(-1)
    a = np.minimum(np.abs(v.astype(np.float64)), 448.0)
    d = np.abs(a[:, None] - vals[None, :])
    best = d.min(1, keepdims=True)
    cand = np.where(d == best, codes[None, :], 1 << 20)
    even = np.where((cand & 1) == 0, cand, 1 << 20).min(1)
    pick = np.where(even < (1 << 20), even, cand.min(1))
    return (np.sign(v) * vals[pick]).astype(np.float32).reshape(shape)


def test_e4m3_rounding_matches_an_independent_table_on_random_values():
    g = torch.Generator().manual_seed(0)
    x = torch.cat([torch.randn(4000, generator=g) * s for s in (1e-3, 0.05, 1.0, 30.0, 300.0)])
    assert np.array_equal(TF8.e4m3(x).numpy(), _np_e4m3(x.numpy()))


def test_weight_quantisation_formula():
    g = torch.Generator().manual_seed(1)
    w = torch.randn(5, 7, 3, 3, generator=g) * torch.tensor([1e-3, 0.1, 1.0, 20.0, 0.0])[:, None, None, None]
    codes, s_w = TF8.quantize_weight(w)
    wn = w.numpy().reshape(5, -1)
    amax = np.abs(wn).max(1)
    s_ref = np.where(amax > 0, amax.astype(np.float32) / np.float32(448.0), np.float32(1.0)).astype(np.float32)
    assert np.array_equal(s_w.numpy(), s_ref)
    ref = _np_e4m3((wn / s_ref[:, None]).astype(np.float32))
    assert np.array_equal(codes.numpy().reshape(5, -1), ref)
    assert np.all(np.abs(codes.numpy().reshape(5, -1)[:4]).max(1) == 448.0)      # the largest weight of a channel maps to 448
    assert s_w[4].item() == 1.0 and codes[4].abs().max().item() == 0.0


def test_epilogue_constants_formula():
    g = torch.Generator().manual_seed(2)
    s_w = torch.rand(64, generator=g) * 1e-3
    bn_scale, bn_shift = torch.randn(64, generator=g), torch.randn(64, generator=g)
    s_in, s_out = 0.0123, 0.456
    scale, shift = quant.epilogue_constants(s_in, s_w, bn_scale, bn_shift, s_out)
    f = np.float32
    ref_scale = ((f(s_in) * s_w.numpy()) * bn_scale.numpy()) / f(s_out)
    ref_shift = bn_shift.numpy() / f(s_out)
    assert scale.dtype == torch.float32 and np.array_equal(scale.numpy(), ref_scale) and np.array_equal(shift.numpy(), ref_shift)
    o_scale, o_shift = TF8.epilogue_constants(s_in, s_w, bn_scale, bn_shift, s_out)
    assert torch.equal(o_scale, scale) and torch.equal(o_shift, shift)
    assert quant.residual_factor(0.3, 0.7) == float(f(0.3) / f(0.7))


def test_activation_scale():
    assert quant.scale_of(torch.tensor(0.0)) == 1.0
    assert quant.scale_of(torch.tensor(3.5)) == float(np.float32(3.5) / np.float32(448.0))
    assert quant.scale_of(torch.tensor(448.0, dtype=torch.bfloat16)) == 1.0
