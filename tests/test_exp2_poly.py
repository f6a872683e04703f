"""The FMA-pipe exp2 of the attention softmax (csrc/attn_tc.cu exp2_poly_f2) restated in fp32 numpy with the
constants read from the source: round-down split x = j + f, degree-3 polynomial on [0, 1), j added to the exponent
field as an integer. Over every input the kernel feeds it (x = S * scale - m_ref <= 8, down to the clamp at -127 and
-inf for masked keys) the relative error stays below 2^-13, a quarter of bf16's half ulp (2^-9) at the very least,
so the bf16 rounding of P stays the dominant error."""
import re
from pathlib import Path

import numpy as np


def _poly_exp2(x):
    src = (Path(__file__).resolve().parents[1] / "marigold_b200" / "csrc" / "attn_tc.cu").read_text()
    c = {int(k): np.float32(float(v)) for k, v in re.findall(r"constexpr float kExp2C(\d) = ([-+0-9.e]+)f;", src)}
    assert sorted(c) == [1, 2, 3]
    x = np.maximum(x.astype(np.float32), np.float32(-127.0))
    magic = np.float32(12582912.0)
    t = (np.floor(x.astype(np.float64)) + 12582912.0).astype(np.float32)      # add.rm: exact for |x| < 2^22
    f = (x - (t - magic)).astype(np.float32)
    q = (c[3] * f + c[2]).astype(np.float32)
    q = (q * f + c[1]).astype(np.float32)
    q = (q * f + np.float32(1.0)).astype(np.float32)
    bits = (q.view(np.uint32).astype(np.uint64) + (t.view(np.uint32).astype(np.uint64) << np.uint64(23))) & np.uint64(0xFFFFFFFF)
    return bits.astype(np.uint32).view(np.float32)


def test_poly_exp2_relative_error_bound():
    rng = np.random.default_rng(0)
    x = np.concatenate([np.linspace(-126.0, 8.0, 2_000_001), rng.uniform(-126.0, 8.0, 1_000_000),
                        np.arange(-126, 9, dtype=np.float64), np.arange(-126, 9) - 2.0 ** -20]).astype(np.float32)
    y = _poly_exp2(x).astype(np.float64)
    ref = np.exp2(x.astype(np.float64))
    rel = np.abs(y / ref - 1.0)
    assert rel.max() <= 2.0 ** -13, rel.max()


def test_poly_exp2_masked_and_underflowing_inputs_are_negligible():
    x = np.array([-np.inf, -1e30, -1000.0, -127.0, -126.5], dtype=np.float32)
    y = _poly_exp2(x)
    assert np.isfinite(y).all() and (y >= 0).all() and (y < 2.0 ** -125).all()
