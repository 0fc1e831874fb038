"""`poly_exp2` (csrc/common.cuh) — the MUFU-free 2^x the attention kernels use for a quarter of their
exponentials.  The constants are read out of the CUDA source and the same float32 / int32
arithmetic is evaluated with numpy, so a changed coefficient or clamp is caught on the CPU."""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "stable-diffusion-1.5-lcm-onnx-rknn2_b200", "csrc", "common.cuh")


def _constants():
    src = open(SRC).read()
    body = src[src.index("float poly_exp2(float x)"):]
    body = body[:body.index("\n}\n")]
    clamp = float(re.search(r"fmaxf\(x, (-?[0-9.]+)f\)", body).group(1))
    magic = float(re.search(r"x \+ ([0-9.]+)f;", body).group(1))
    c3, c2 = map(float, re.search(r"fmaf\(([0-9.eE+-]+)f, f, ([0-9.eE+-]+)f\)", body).groups())
    c1, c0 = [float(m) for m in re.findall(r"fmaf\(p, f, ([0-9.eE+-]+)f\)", body)]
    assert "<< 23" in body
    return clamp, magic, (c0, c1, c2, c3)


def _packed_constants():
    """The same constants from the packed (f32x2) copy that attn_pp_kernel (csrc/attention_pp.cu, the SD1.5 head
    dim 40 path) inlines: clamp, rounding constant, -1 of the Cody-Waite step and the four coefficients, each pair
    with the same value in both lanes."""
    src = open(os.path.join(os.path.dirname(SRC), "attention_pp.cu")).read()
    body = src[src.index("packed 2^x on the FMA / ALU pipes"):]
    body = body[:body.index("} else {")]
    clamps = {float(v) for v in re.findall(r"fmaxf\(x[01], (-?[0-9.]+)f\)", body)}
    assert len(clamps) == 1, clamps
    pairs = re.findall(r"f2_pack\((-?[0-9.eE+-]+)f, (-?[0-9.eE+-]+)f\)", body)
    assert all(a == b for a, b in pairs), pairs
    vals = [float(a) for a, _ in pairs]
    # r = x + magic, t = r - magic, f = t * -1 + x, then c3 * f + c2, * f + c1, * f + c0
    assert len(vals) == 7, vals
    magic, neg_magic, neg_one, c3, c2, c1, c0 = vals
    assert neg_magic == -magic and neg_one == -1.0, vals
    assert "<< 23" in body
    return clamps.pop(), magic, (c0, c1, c2, c3)


def _poly_exp2(x, clamp, magic, c):
    f32 = np.float32
    x = np.maximum(x.astype(f32), f32(clamp))
    r = (x + f32(magic)).astype(f32)
    f = (x - (r - f32(magic)).astype(f32)).astype(f32)
    p = (f32(c[3]) * f + f32(c[2])).astype(f32)
    p = (p * f + f32(c[1])).astype(f32)
    p = (p * f + f32(c[0])).astype(f32)
    bits = (p.view(np.int32).astype(np.int64) + ((r.view(np.int32).astype(np.int64) << 23) & 0xFFFFFFFF)) & 0xFFFFFFFF
    return bits.astype(np.uint32).view(f32)


def test_poly_exp2_matches_exp2_over_the_softmax_range():
    clamp, magic, c = _constants()
    assert magic == 1.5 * 2 ** 23 and -126.0 < clamp <= -100.0
    # the kernel feeds x = s * scale * log2(e) - m_run: <= 8 (lazy running max) and unbounded below
    x = np.linspace(-140.0, 9.0, 1_500_001).astype(np.float32)
    y = _poly_exp2(x, clamp, magic, c)
    ref = 2.0 ** np.maximum(x.astype(np.float64), clamp)
    rel = np.abs(y / ref - 1.0)
    assert np.isfinite(y).all() and (y > 0).all()
    assert rel.max() <= 1e-4, rel.max()                  # bf16 rounding of P is 2e-3
    # monotone up to the polynomial's own error at the seams f = +-0.5
    assert (np.diff(y.astype(np.float64)) >= -2e-4 * y[1:]).all()


def test_poly_exp2_edge_cases():
    clamp, magic, c = _constants()
    x = np.array([-np.inf, -1e30, clamp, 0.0, 1.0, -1.0, 0.5, -0.5, 8.0, 8.49], dtype=np.float32)
    y = _poly_exp2(x, clamp, magic, c)
    assert np.isfinite(y).all()
    assert y[0] == y[1] == y[2] and 0 < y[0] < 1e-30       # masked keys (-inf) vanish in P
    assert abs(y[3] - 1.0) < 1e-4 and abs(y[4] - 2.0) < 2e-4 and abs(y[5] - 0.5) < 5e-5
    assert abs(y[8] - 256.0) < 256 * 1e-4
    # the row maximum gets P = 1.0 exactly after the bf16 rounding (8 mantissa bits)
    assert np.float32(y[3]).view(np.uint32) + 0x8000 >> 16 == 0x3F80


def test_attn_pp_packed_copy_matches_common():
    """attn_pp_kernel's inlined packed 2^x must be the polynomial pinned above, constant for constant."""
    assert _packed_constants() == _constants()
