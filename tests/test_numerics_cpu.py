"""CPU re-statements (numpy, float32 arithmetic where the kernels use it) of two pieces of device arithmetic whose error
bounds DESIGN.md / the kernel comments state - so that the bounds are checked, not only claimed:
  * the exact-erf GELU polynomial of the fc1 epilogue (gemm_tc.cu: gelu_erf2),
  * the shifted per-slice LayerNorm statistics and their combination in the consuming GEMM (gemm_tc.cu epilogue)."""
import math

import numpy as np

f32 = np.float32


def test_gelu_polynomial_matches_exact_erf_gelu():
    # gemm_tc.cu: gelu(x) = x * (0.5 + xc * q(xc^2)), xc = clamp(x, -4.5, 4.5), q of degree 9, fp32 Horner
    coef = [-1.3369040159e-12, 1.6336444415e-10, -8.9213697499e-09, 2.8944761772e-07, -6.2733902842e-06, 9.7063541348e-05,
            -1.1183810776e-03, 9.8202145566e-03, -6.6317755718e-02, 3.9887377948e-01]
    x = np.linspace(-8.0, 8.0, 200001).astype(f32)
    xc = np.clip(x, f32(-4.5), f32(4.5))
    u = (xc * xc).astype(f32)
    q = np.full_like(u, f32(coef[0]))
    for c in coef[1:]:
        q = (q * u + f32(c)).astype(f32)
    got = (x * (xc * q + f32(0.5))).astype(f32)
    ref = np.array([0.5 * v * (1.0 + math.erf(v / math.sqrt(2.0))) for v in x.astype(np.float64)])
    err = np.abs(got.astype(np.float64) - ref)
    assert err.max() < 1.0e-4                                   # stated: max |error| 7.4e-5 (at |x| ~ 4.46 where gelu ~ 4.46)
    assert err[np.abs(x) < 3.0].max() < 1.0e-5                  # stated: < 1e-5 for |x| < 3
    # relative to the 16-bit rounding of the output it feeds: within one fp16 rounding (4.9e-4) wherever |gelu| > 1e-2 (the worst
    # case is the small negative lobe, gelu(-2.5) = -0.0155 with an absolute error of 6e-6), below 1e-4 for positive x
    big = np.abs(ref) > 1e-2
    assert (err[big] / np.abs(ref[big])).max() < 4.9e-4
    pos = x > 0.05
    assert (err[pos] / np.abs(ref[pos])).max() < 1.0e-4


def _producer_partials(row, parts):
    """gemm_tc.cu producer epilogue: per column slice, K = first value, sums of (x - K) and (x - K)^2 in fp32,
    partial = (n*K + s1, s2 - s1^2/n)."""
    out = []
    for sl in np.split(row.astype(f32), parts):
        K = sl[0]
        d = (sl - K).astype(f32)
        s1 = f32(0.0)
        s2 = f32(0.0)
        for v in d:                                             # sequential fp32 accumulation, as one thread does it
            s1 = f32(s1 + v)
            s2 = f32(s2 + v * v)
        n = f32(len(sl))
        out.append((f32(n * K + s1), f32(max(s2 - s1 * s1 / n, f32(0.0)))))
    return out


def _consumer_stats(partials, C, eps):
    """gemm_tc.cu consumer: mean = sum(sum_p)/C; var = [sum(M2_p) + n_p * sum((sum_p/n_p - mean)^2)] / C."""
    n_p = f32(C / len(partials))
    s1 = f32(0.0)
    for sp, _ in partials:
        s1 = f32(s1 + sp)
    mean = f32(s1 / f32(C))
    m2 = f32(0.0)
    for sp, mp in partials:
        dm = f32(sp / n_p - mean)
        m2 = f32(m2 + mp + n_p * dm * dm)
    return mean, f32(1.0) / np.sqrt(f32(m2 / f32(C) + f32(eps)))


def test_shifted_layernorm_statistics_combine_exactly_and_survive_large_means():
    rng = np.random.default_rng(0)
    for C, parts in ((192, 4), (192, 2), (384, 4), (384, 8), (768, 12), (768, 6)):
        for mean0, std0 in ((0.0, 1.0), (3.0, 0.5), (200.0, 0.25), (-1000.0, 0.1)):
            row = (rng.standard_normal(C) * std0 + mean0).astype(np.float16).astype(np.float64)   # the rounded 16-bit row the consumer reads
            mean_ref, var_ref = row.mean(), row.var()
            mean, rstd = _consumer_stats(_producer_partials(row, parts), C, 1e-6)
            rstd_ref = 1.0 / math.sqrt(var_ref + 1e-6)
            assert abs(float(mean) - mean_ref) <= 2e-6 * max(1.0, abs(mean_ref)), (C, parts, mean0)
            if var_ref > 1e-12:
                assert abs(float(rstd) - rstd_ref) / rstd_ref < 2e-4, (C, parts, mean0, std0, float(rstd), rstd_ref)
    # what the shift buys: the single-pass form E[x^2] - mean^2 in fp32 loses the variance of such a row entirely
    row = (rng.standard_normal(192) * 0.25 + 1000.0).astype(np.float16).astype(np.float64)
    x = row.astype(f32)
    naive_var = f32(np.sum(x * x, dtype=f32) / f32(192)) - f32(np.sum(x, dtype=f32) / f32(192)) ** 2
    _, rstd = _consumer_stats(_producer_partials(row, 4), 192, 1e-6)
    good = abs(float(rstd) - 1.0 / math.sqrt(row.var() + 1e-6)) * math.sqrt(row.var() + 1e-6)
    bad = abs(float(naive_var) - row.var()) / row.var()
    assert good < 1e-3 and bad > 0.05, (good, bad)
