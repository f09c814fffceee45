"""CPU: the hand-rolled device arithmetic of the kernels, restated operation by operation in numpy float32
(fused multiply-adds evaluated in float64 and rounded once, as the hardware does), checked against libm:

* the degree-3 exp2 polynomial the attention softmax runs on the FMA pipe for a quarter of the exponentials
  (attention_common.cuh `exp2_poly2`) -- claimed relative error 7.5e-5, far below the
  resolution of the 16-bit P operand (bf16: 3.9e-3, fp16: 4.9e-4);
* the two-constant Cody-Waite reduction in front of `__sincosf` for the RoPE angles (rowops.cu `fast_sincos`);
* the LDR quantisation rule of `rfb_ldr_quantize` mode 0 (dpt.cu) against the reference CLIs' numpy expression.

The constants are read out of the .cu sources, so the test follows the code."""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "renderformer_b200", "csrc")
f32 = np.float32


def _fma(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(f32)


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _poly_constants(src, fn):
    body = src[src.index(fn):]
    body = body[:body.index("\n}\n")]
    magic = f32(re.search(r"pack2f\((\d+\.\d+)f, \1f\)", body).group(1))
    coef = [f32(m) for m in re.findall(r"pack2f\((0\.\d+)f, \1f\)", body)]
    clamp = f32(re.search(r"fmaxf\(lo2f\(t2\), (-\d+\.\d+)f\)", body).group(1))
    return magic, coef, clamp


def _exp2_poly(t, magic, coef, clamp):
    """exp2_poly2: t = n + f with n = round(t); 2^f by Horner in f; 2^n by adding n to the exponent field
    (r = t + 1.5 * 2^23 keeps n in the low mantissa bits of r)."""
    t = np.maximum(t.astype(f32), clamp)
    r = (t + magic).astype(f32)
    n = (r - magic).astype(f32)
    f = _fma(n, np.full_like(n, -1.0), t)
    c3, c2, c1, c0 = coef
    p = _fma(f, np.full_like(f, c3), np.full_like(f, c2))
    p = _fma(p, f, np.full_like(f, c1))
    p = _fma(p, f, np.full_like(f, c0))
    bits = p.view(np.uint32) + (r.view(np.uint32) << np.uint32(23))
    return bits.view(f32)


def test_softmax_exp2_polynomial_accuracy():
    name = "attention_common.cuh"
    magic, coef, clamp = _poly_constants(_src(name), "void exp2_poly2(")
    assert magic == f32(12582912.0) and len(coef) == 4 and clamp == f32(-126.0), name
    t = np.concatenate([np.linspace(-126.0, 0.0, 2_000_001), -np.arange(0.0, 127.0), [-0.5, -1.5, -125.5]]).astype(f32)
    got = _exp2_poly(t, magic, coef, clamp).astype(np.float64)
    want = np.exp2(t.astype(np.float64))
    rel = np.abs(got - want) / want
    # below 2^-125 the polynomial's value (< 1) times 2^n leaves the normal range: the exponent-field trick then
    # yields a denormal-coded number of the right magnitude only (1e-38: a probability that is zero in any sum)
    normal = t >= f32(-125.0)
    assert rel[normal].max() <= 1.0e-4, (name, rel[normal].max())   # claimed 7.5e-5 (+ fp32 rounding)
    assert rel[normal].max() < 0.25 * 2.0 ** -11                      # well under half an ulp of fp16, 16x under bf16's
    assert (got[~normal] >= 0).all() and (got[~normal] <= 2.0 ** -125).all()
    assert (got <= 1.0 + 1e-4).all() and (got > 0).all()   # probabilities stay in (0, 1]
    # inputs below the clamp (masked keys arrive as -inf) give the smallest normal, never NaN / negative
    low = _exp2_poly(np.array([-1e4, -np.inf], dtype=f32), magic, coef, clamp)
    assert np.isfinite(low).all() and (low >= 0).all() and (low <= 1.2e-38).all()
    # monotone on a fine grid around every integer boundary (the n / f split must not tear the curve)
    edge = (np.arange(-125, 0)[:, None] + np.linspace(-0.5, 0.5, 2001)[None, :]).astype(f32).reshape(-1)
    y = _exp2_poly(np.sort(edge), magic, coef, clamp)
    assert (np.diff(y.astype(np.float64)) >= -1e-4 * y[1:]).all()


def test_rope_angle_reduction_constants():
    src = _src("rowops.cu")
    body = src[src.index("void fast_sincos("):]
    body = body[:body.index("__sincosf")]
    inv2pi = f32(re.search(r"x \* (0\.\d+)f", body).group(1))
    hi, lo = [np.float64(m) for m in re.findall(r"fmaf\(k, (-?\d\.\d+(?:e-?\d+)?)f", body)]
    assert abs(float(inv2pi) - 1.0 / (2 * np.pi)) < 1e-8
    assert f32(hi) == f32(-2 * np.pi)                                   # the fp32 nearest to 2 pi, negated
    assert abs((-float(f32(hi)) - float(f32(lo))) - 2 * np.pi) < 1e-13   # hi + lo carries 2 pi to ~48 bits
    # angles seen by the kernels: |position| <~ 2 (scene in the unit sphere, camera within a few units) times the
    # largest RoPE frequency 5.0, with a wide margin
    x = np.concatenate([np.linspace(-100, 100, 1_000_001), [0.0, np.pi, -np.pi, 2 * np.pi, 50 * np.pi]]).astype(f32)
    k = np.rint((x * inv2pi).astype(f32)).astype(f32)
    r = _fma(k, np.full_like(k, f32(hi)), x)
    r = _fma(k, np.full_like(k, f32(lo)), r)
    assert np.abs(r).max() <= np.pi * (1 + 1e-6)
    # reduced angle == x mod 2 pi to ~1e-6 absolute, so sin / cos of it match to the same order
    err_s = np.abs(np.sin(r.astype(np.float64)) - np.sin(x.astype(np.float64)))
    err_c = np.abs(np.cos(r.astype(np.float64)) - np.cos(x.astype(np.float64)))
    assert max(err_s.max(), err_c.max()) <= 2e-6


def test_ldr_rule_matches_numpy_expression():
    """dpt.cu mode 0: (uint8)(__fmul_rn(fminf(fmaxf(x, 0), 1), 255)) == (np.clip(x, 0, 1) * 255).astype(np.uint8)
    (batch_infer.py:153-157) for every fp32 in [0, 1] that lands near an integer boundary, and outside."""
    k = np.arange(0, 256, dtype=np.float64)
    edges = (k / 255.0).astype(f32)
    xs = np.concatenate([np.nextafter(edges, f32(-1)), edges, np.nextafter(edges, f32(2)),
                         np.array([-3.0, -0.0, 1.0, 1.5, 5000.0], dtype=f32)])
    dev = np.trunc((np.minimum(np.maximum(xs, f32(0)), f32(1)) * f32(255)).astype(f32)).astype(np.uint8)  # fp32 product, truncation
    ref = (np.clip(xs, 0, 1) * 255).astype(np.uint8)
    assert np.array_equal(dev, ref)
    src = _src("dpt.cu")
    assert "__fmul_rn(fminf(fmaxf(r, 0.f), 1.f), 255.f)" in src
