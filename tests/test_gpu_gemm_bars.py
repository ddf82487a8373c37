"""The tcgen05 GEMM and its fused epilogues against an fp64 reference, with bars tight enough to see a dropped k-block,
row or column.

test_gpu_kernels.py compares these kernels with an fp32 torch result at 2e-2 x max|ref| (about 10x the bf16 rounding
floor), so an output off by 0.2 % or missing one k of K = 576 passes there. Here every case is checked against

  * relative L2          ||out - ref|| / ||ref||
  * max |out - ref| / rms(ref)
  * gain |<out - ref, ref>| / <ref, ref>   (bf16 outputs only)

The reference is the exact float64 product of the bf16 operands the kernel receives, followed by bias, activation
(erf GELU), residual, LayerNorm or the up-scaling epilogue in float64. The emulated floor is what a correct kernel must
produce: the float64 product rounded to fp32 (the TMEM accumulator), the epilogue in fp32 with the kernel's own GELU
formula (common.cuh gelu_erf: tanh form, here with an exact tanh) and sigmoid, then rounding to the output dtype. Every
case asserts that the floor is within half of each bar, so no bar asks for more than the arithmetic allows.

The gain bar exists because bf16 rounding alone is ~1.1e-3 relative L2: a relative L2 bar that keeps the floor under
half of it cannot see an output scaled by 0.998 (2e-3 in quadrature with the floor is 2.3e-3). Rounding to nearest is
unbiased, so the floor's gain is ~1e-5 and a 0.2 % scale shows as 2e-3.

GELU routes: tanh.approx.f32 (MUFU.TANH) has a relative error of at most 2^-10.987 (PTX ISA), and the tanh form differs
from erf GELU by up to ~2e-4. Both are modelled per element as an envelope
  env = |gelu_tanh_form(x) - gelu_erf(x)| + 0.5 |x| (|tanh(.)| 2^-10.987 + 2^-20)
(summed with |hyper| weights through UP2's dot product); the L2 and max bars apply to max(|out - ref| - env, 0).

Inputs make every k, row and column count: "flat" random operands; "kbeacon" puts a 16x column of A (one per group of
rows, +-16) against a +-1 column of W at k = 0, K - 1, both sides of the 16-k steps of the first k-block, of every
k-block edge up to the 9th (the operand ring holds at most 8 stages, so this includes where it wraps) and of the last
k-block edge: a dropped k-block, k-step or ragged K tail moves those rows by ~3x rms; "markers" scales every row of A
and of W by a distinct factor in [1, 1.5) so a row or column written to the wrong place (also across the two CTAs of
a pair tile) shows; "hotres" makes the residual 100x the product (a residual row m instead of m % res_mod, or the
wrong residual dtype); LN cases add "offset rows" with |mean| / std of 64 and 256. A, W and the residual are views into
wider buffers whose unused columns and rows past M / N hold +-3e4; the output goes into a buffer with extra columns
(ldo > N) and one extra pair tile of rows, pre-filled with a NaN bit pattern that must survive bit for bit.

Bars: see BF16_BARS / F32_BARS. The CPU tests at the end pin that the floor sits at most at half of each bar on every
route's shape class and that the defects the bars exist for fail them. The GPU cases of this file take ~15 s on a B200
(the SM-budget test, with its two child processes, ~10 s of that).
"""
import math
import os
import subprocess
import sys
import tempfile

import pytest
import torch

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (relative L2, max |err| / rms(ref), gain or None). Measured on an NVIDIA B200 (1000 W power limit) over this file's
# GPU cases:
# bf16 outputs: every kernel result equals its emulated floor to the printed digits: relative L2 1.2e-3-2.0e-3 (2.0e-3
# on 100 outputs of one row), max 0.004-0.029 x rms, gain <= 2.8e-4 (a sigmoid output of 64 x 272 values: positive
# outputs, few of them); every bar sits at least 2x above the worst floor.
# fp32 outputs: kernels <= 8.6e-6 relative L2 and <= 3.3e-5 x rms max (fp32 accumulation over K = 4608, 6-term split
# product, UP2's dot product); floors <= 1.2e-5 / 6.4e-5, the largest on LN rows with |mean| / std ~ 256, where the fp32
# sum x = acc + bias + residual alone loses |mean| x 2^-24. A one-pass fp32 variance of such rows (sumsq / N - mean^2,
# what the LN epilogue computed before it summed x - x0) measured 2.1e-4-3.0e-4 relative L2 and 2.5e-3-4.1e-3 x rms at
# |mean| / std = 64; with the shifted sums 2.1e-6 / <= 1.0e-5 there, 8.4e-6 / <= 3.1e-5 at 256.
# A single row (M = 1) has too few outputs for the L2 bar to sit far from bf16 rounding, hence 4e-3 rather than 3e-3.
BF16_BARS = (4e-3, 0.08, 1e-3)
F32_BARS = (4e-5, 4e-4, None)

SENT = 3e4
NAN_BITS = {BF16: 0x7FA5, F32: 0x7FA5A5A5}
TANH_APPROX_REL = 2.0 ** -10.987
ACT_NONE, ACT_GELU, ACT_RELU, ACT_SIGMOID = 0, 1, 2, 3


# ------------------------------------------------------------------------------------------------------------------
# Activations: exact (float64), the kernel's formulas (fp32 floor) and the modelled GELU error
# ------------------------------------------------------------------------------------------------------------------
def _gelu_tanh_form(x):
    """common.cuh gelu_erf with an exact tanh, in x's dtype."""
    z = x * 0.70710678118654752440
    t = torch.tanh(z * (z * z * 0.0997927 + 1.12967583))
    hx = 0.5 * x
    return hx * t + hx


def _gelu_env(x):
    """Modelled |kernel GELU - erf GELU| at pre-activation x (float64)."""
    z = x * 0.70710678118654752440
    t = torch.tanh(z * (z * z * 0.0997927 + 1.12967583))
    form = (_gelu_tanh_form(x) - 0.5 * x * (1.0 + torch.erf(z))).abs()
    return form + 0.5 * x.abs() * (t.abs() * TANH_APPROX_REL + 2.0 ** -20)


def _act_exact(x, act):
    if act == ACT_GELU:
        return 0.5 * x * (1.0 + torch.erf(x * 0.70710678118654752440))
    if act == ACT_RELU:
        return x.clamp_min(0)
    if act == ACT_SIGMOID:
        return torch.sigmoid(x)
    return x


def _act_floor(x32, act):
    if act == ACT_GELU:
        return _gelu_tanh_form(x32)
    if act == ACT_RELU:
        return x32.clamp_min(0)
    if act == ACT_SIGMOID:
        return 1.0 / (1.0 + torch.exp(-x32))
    return x32


# ------------------------------------------------------------------------------------------------------------------
# Errors and bars
# ------------------------------------------------------------------------------------------------------------------
def _errors(out, ref, env=None):
    e = out.to(F64) - ref
    d = e.abs() if env is None else (e.abs() - env).clamp_min(0)
    rr = ref.pow(2).sum()
    rms = (rr / ref.numel()).sqrt()
    # the gain of a few outputs is as noisy as their rounding: it is measured from 4096 outputs on
    gain = ((e * ref).sum() / rr).abs().item() if ref.numel() >= 4096 else float("nan")
    return (d.norm() / rr.sqrt()).item(), (d.max() / rms).item(), gain


def _fails(errs, bars):
    return errs[0] > bars[0] or errs[1] > bars[1] or (bars[2] is not None and errs[2] > bars[2])


def assert_close(out, ref, floor, case, fp32, env=None):
    """All bars on the kernel output, and the emulated floor within half of each bar."""
    bars = F32_BARS if fp32 else BF16_BARS
    assert out.shape == ref.shape, (out.shape, ref.shape)
    assert torch.isfinite(out).all(), f"{case}: non-finite output"
    k, f = _errors(out, ref, env), _errors(floor, ref, env)
    print(f"\n[bars] {case}: rel_l2 {k[0]:.2e} max/rms {k[1]:.2e} gain {k[2]:.1e} | "
          f"floor {f[0]:.2e} {f[1]:.2e} {f[2]:.1e}")
    half = tuple(None if b is None else b / 2 for b in bars)
    assert not _fails(f, half), f"{case}: emulated floor {f} above half the bars {bars}"
    assert not _fails(k, bars), f"{case}: rel_l2 {k[0]:.3e} max/rms {k[1]:.4f} gain {k[2]:.2e} (bars {bars})"


# ------------------------------------------------------------------------------------------------------------------
# Inputs
# ------------------------------------------------------------------------------------------------------------------
def k_positions(K):
    """k = 0, K - 1 and both sides of the 16-k steps of the first k-block, of every 64-k-block edge up to the 9th and of
    the last k-block edge, without duplicates."""
    edges = [16, 32, 48] + [64 * s for s in range(1, 10)] + [64 * ((K - 1) // 64)]
    pos = [0, K - 1]
    for e in edges:
        pos += [e - 1, e]
    out = []
    for p in pos:
        if 0 < p < K or p == 0:
            if p not in out:
                out.append(p)
    return out


def _frac_scale(n, phi, device):
    i = torch.arange(n, device=device, dtype=F64)
    return (1.0 + 0.5 * torch.frac(i * phi + 0.1)).float()


def _operands(kind, M, N, K, gen, device):
    a = torch.randn(M, K, generator=gen, device=device)
    w = torch.randn(N, K, generator=gen, device=device) / math.sqrt(K)
    if kind == "kbeacon":
        pos = k_positions(K)
        G = len(pos)
        grp = torch.arange(M, device=device) % G
        sa = torch.where(torch.rand(M, generator=gen, device=device) < 0.5, 16.0, -16.0)
        for g, k in enumerate(pos):
            sel = grp == g
            a[sel, k] = sa[sel]
            w[:, k] = torch.where(torch.rand(N, generator=gen, device=device) < 0.5, 1.0, -1.0)
    elif kind == "markers":
        a *= _frac_scale(M, 0.6180339887498949, device)[:, None]
        w *= _frac_scale(N, 0.7548776662466927, device)[:, None]
    else:
        assert kind in ("flat", "hotres"), kind
    return a, w


def _guarded(x, rows_extra, cols_extra, dtype, gen):
    """x [R, C] as a view into a [R + rows_extra, C + cols_extra] buffer whose other cells hold +-3e4."""
    R, C = x.shape
    buf = torch.where(torch.rand(R + rows_extra, C + cols_extra, generator=gen, device=x.device) < 0.5, SENT, -SENT)
    buf = buf.to(dtype)
    buf[:R, :C] = x.to(dtype)
    return buf[:R, :C]


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == BF16 else torch.int32)


def _out_buffer(M, N, dtype, device, extra_cols=True):
    """Output buffer with 8 (bf16) / 4 (fp32) extra columns and 256 extra rows, filled with a NaN bit pattern."""
    cols = N + ((8 if dtype == BF16 else 4) if extra_cols else 0)
    it = torch.int16 if dtype == BF16 else torch.int32
    return torch.full((M + 256, cols), NAN_BITS[dtype], dtype=it, device=device).view(dtype)


def assert_guard_intact(buf, M, N, case):
    bits = _bits(buf)
    guard = torch.ones(bits.shape, dtype=torch.bool, device=bits.device)
    guard[:M, :N] = False
    bad = (bits[guard] != NAN_BITS[buf.dtype]).sum().item()
    assert bad == 0, f"{case}: {bad} guard cells outside the [{M}, {N}] output were written"


class Std:
    """One sb_gemm_bf16 problem: out = act(alpha * a @ w^T + bias) + res[m % res_mod or m]."""

    def __init__(self, M, N, K, bn=0, out="bf16", act=0, bias=False, res=None, res_mod=0, alpha=1.0, route=""):
        self.M, self.N, self.K, self.bn, self.act, self.bias, self.res, self.res_mod, self.alpha = \
            M, N, K, bn, act, bias, res, res_mod, alpha
        self.out = BF16 if out == "bf16" else F32
        self.route = route

    @property
    def id(self):
        r = f"-res{self.res}" + (f"mod{self.res_mod}" if self.res_mod else "") if self.res else ""
        return (f"{self.route}-M{self.M}-N{self.N}-K{self.K}-{'bf16' if self.out == BF16 else 'f32'}-act{self.act}"
                f"{'-bias' if self.bias else ''}{r}{'-alpha' + str(self.alpha) if self.alpha != 1.0 else ''}")


def std_inputs(c, kind, seed, device="cuda"):
    gen = torch.Generator(device=device).manual_seed(seed)
    a, w = _operands(kind, c.M, c.N, c.K, gen, device)
    d = dict(a=_guarded(a, 128, 24, BF16, gen), w=_guarded(w, 64, 24, BF16, gen), bias=None, res=None, res_rows=None)
    if c.bias:
        d["bias"] = 0.5 * torch.randn(c.N, generator=gen, device=device)
    if c.res:
        R = c.res_mod if c.res_mod else c.M
        r = torch.randn(R, c.N, generator=gen, device=device) * (100.0 if kind == "hotres" else 1.0)
        d["res"] = _guarded(r, 32, 8, BF16 if c.res == "bf16" else F32, gen)
        # what follows the res_mod rows in memory (a kernel reading row m instead of m % res_mod would see other data)
        d["res_rows"] = torch.randn(c.M, c.N, generator=gen, device=device)
    return d


def std_reference(c, d, rows=None, defect=None):
    """(exact fp64, emulated floor as fp64 values of the output dtype, GELU envelope or None) for output rows `rows`."""
    a, w = d["a"], d["w"]
    if rows is not None:
        a = a[rows]
    a64, w64 = a.to(F64), w.to(F64)
    acc = a64 @ w64.t()
    acc_floor = acc
    if defect in ("drop_kblock", "drop_partial_tail"):  # the second k-block, or the last k-block's last k-step(s)
        a64 = a64.clone()
        a64[:, slice(64, 128) if defect == "drop_kblock" else slice((c.K - 1) // 64 * 64 + (16 if c.K <= 64 else 0), None)] = 0
        acc_floor = a64 @ w64.t()
    m = torch.arange(c.M, device=acc.device) if rows is None else rows
    b64 = d["bias"].to(F64) if d["bias"] is not None else torch.zeros(c.N, dtype=F64, device=acc.device)
    x = c.alpha * acc + b64
    ref = _act_exact(x, c.act)
    env = _gelu_env(x) if c.act == ACT_GELU else None
    # floor: fp32 accumulator, fma(acc, alpha, bias), activation, + residual, round
    acc32 = acc_floor.to(F32)
    if defect == "bf16_acc":
        acc32 = acc32.to(BF16).to(F32)
    b32 = b64.to(F32)
    if defect == "bias_missing_last_tile":
        b32 = b32.clone()
        b32[256:] = 0
    y32 = _act_floor((acc32.to(F64) * c.alpha + b32.to(F64)).to(F32), c.act)
    if d["res"] is not None:
        rr = m % c.res_mod if c.res_mod else m
        res = d["res"][rr]
        ref = ref + res.to(F64)
        if defect == "residual_row_m":  # rows past res_mod read what follows the residual rows
            res = torch.where((m >= c.res_mod)[:, None], d["res_rows"][m].to(res.dtype), res)
        y32 = y32 + res.to(F32)
    floor = y32.to(c.out).to(F64)
    if defect == "scale_0.998":
        floor = (y32 * 0.998).to(c.out).to(F64)
    elif defect == "row_moved_in_warp":  # row 5 of the first 32-row slice written with row 6's values
        floor = floor.clone()
        floor[5] = floor[6]
    return ref, floor, env


def run_std(ops, c, d):
    buf = _out_buffer(c.M, c.N, c.out, d["a"].device)
    out = ops.gemm(d["a"], d["w"], d["bias"], c.act, d["res"], c.res_mod, c.out, out=buf[:c.M, :c.N], alpha=c.alpha,
                   force_bn=c.bn)
    return out, buf


# Route matrix. Single CTA: force_bn 64 / 128 / 192 / 256 ("cta<bn>"); CTA pair: force_bn -128 / -192 / -256
# ("pair<bn>", 256-row tiles, M >= 4096, N >= 128). The STD epilogue is "staged" (coalesced through shared memory) unless
# N % 16 != 0, res_mod % 32 != 0 or a pitch is not a multiple of 16 bytes ("scalar"); a residual of the output's dtype
# is staged in place ("alias"), another one separately ("sep"); "rb1" / "rb2" = residual staging buffers (one when
# K >= 1152 frees a pipeline stage, or when the 256-wide ring would be shallower than 3 stages); "vec" = the whole bias
# vector is staged once (several column tiles); "split" = both epilogue warp sets drain every tile (K >= 512).
STD_CASES = [
    Std(1, 272, 32, 64, "bf16", route="cta64-staged-vec"),
    Std(64, 32, 72, 64, "f32", ACT_SIGMOID, bias=True, alpha=0.5, route="cta64-staged"),
    Std(4097, 100, 200, 128, "bf16", ACT_GELU, bias=True, route="cta128-scalar"),
    Std(4225, 4, 4608, 64, "f32", bias=True, res="f32", route="cta64-scalar-res-split"),
    Std(4225, 272, 72, 256, "f32", ACT_RELU, bias=True, res="f32", res_mod=1000, route="cta256-scalar-resmod"),
    Std(1, 100, 200, 64, "bf16", bias=True, res="f32", route="cta64-scalar-res"),
    Std(4097, 272, 200, 192, "bf16", ACT_RELU, bias=True, res="bf16", res_mod=1024, route="cta192-staged-alias-rb2-vec"),
    Std(4097, 272, 200, 128, "f32", bias=True, res="bf16", alpha=-0.75, route="cta128-staged-sep-rb2-vec"),
    Std(70000, 272, 4608, 192, "f32", bias=True, res="f32", route="cta192-staged-alias-rb1-vec-split"),
    Std(4225, 272, 4608, 256, "bf16", ACT_GELU, bias=True, res="f32", route="cta256-staged-sep-rb1-vec-split"),
    Std(64, 272, 4608, 128, "bf16", ACT_SIGMOID, res="bf16", res_mod=32, route="cta128-staged-alias-rb1-vec-split"),
    Std(70000, 32, 32, 64, "bf16", ACT_GELU, bias=True, alpha=1.5, route="cta64-staged"),
    Std(4097, 272, 200, -128, "bf16", ACT_GELU, bias=True, route="pair128-vec"),
    Std(4097, 128, 200, -128, "f32", bias=True, route="pair128"),
    Std(4224, 272, 4608, -192, "f32", bias=True, res="f32", res_mod=2048, route="pair192-res-vec"),
    Std(4225, 272, 72, -256, "bf16", ACT_RELU, bias=True, res="bf16", route="pair256-res-vec"),
    Std(4351, 272, 32, -256, "f32", ACT_SIGMOID, alpha=2.0, route="pair256-vec"),
    Std(70000, 272, 4608, -128, "bf16", bias=True, route="pair128-vec"),
]


def _kinds(c):
    return ["flat", "kbeacon", "markers"] + (["hotres"] if c.res else [])


# ------------------------------------------------------------------------------------------------------------------
# GEMM-LN
# ------------------------------------------------------------------------------------------------------------------
def ln_inputs(M, N, K, res, res_mod, offset, seed, device="cuda"):
    gen = torch.Generator(device=device).manual_seed(seed)
    a, w = _operands("flat", M, N, K, gen, device)
    d = dict(a=_guarded(a, 128, 24, BF16, gen), w=_guarded(w, 64, 24, BF16, gen),
             bias=0.5 * torch.randn(N, generator=gen, device=device),
             gamma=1.0 + 0.1 * torch.randn(N, generator=gen, device=device),
             beta=0.1 * torch.randn(N, generator=gen, device=device), res=None)
    R = res_mod if res_mod else M
    r = torch.randn(R, N, generator=gen, device=device)
    if offset:  # rows of std ~1.5 (product 1, bias 0.5, residual 1) shifted by +-offset std
        r += 1.5 * offset * torch.where(torch.rand(R, 1, generator=gen, device=device) < 0.5, 1.0, -1.0)
    d["res"] = _guarded(r, 32, 8, BF16 if res == "bf16" else F32, gen)
    return d


def _ln_onepass_stats(x32):
    """mean and variance of a one-pass LN epilogue on the raw values: per 16-column chunk two interleaved fp32
    partial sums of x and x^2 (packed pairs), chunk sums added into fp32 row totals, var = sumsq / N - mean^2."""
    M, N = x32.shape
    s = torch.zeros(M, dtype=F32, device=x32.device)
    q = torch.zeros(M, dtype=F32, device=x32.device)
    for c0 in range(0, N, 16):
        s2 = torch.zeros(M, 2, dtype=F32, device=x32.device)
        q2 = torch.zeros(M, 2, dtype=F32, device=x32.device)
        for j in range(8):
            ff = x32[:, c0 + 2 * j:c0 + 2 * j + 2]
            s2 = s2 + ff
            q2 = (ff.to(F64) * ff + q2).to(F32)
        s = s + (s2[:, 0] + s2[:, 1])
        q = q + (q2[:, 0] + q2[:, 1])
    mean = s / N
    var = (q / N - mean * mean).clamp_min(0)
    return mean, var


def ln_reference(d, M, N, res_mod, eps, out_dtype, defect=None):
    acc = d["a"].to(F64) @ d["w"].to(F64).t()
    m = torch.arange(M, device=acc.device)
    res = d["res"][m % res_mod if res_mod else m]
    x = acc + d["bias"].to(F64) + res.to(F64)
    mu = x.mean(1, keepdim=True)
    var = (x - mu).pow(2).mean(1, keepdim=True)
    ref = (x - mu) / torch.sqrt(var + eps) * d["gamma"].to(F64) + d["beta"].to(F64)
    x32 = (acc.to(F32) + d["bias"]) + res.to(F32)
    if defect == "onepass_variance":
        mean32, var32 = _ln_onepass_stats(x32)
    else:
        mean32 = x32.mean(1)
        var32 = (x32 - mean32[:, None]).pow(2).mean(1)
    rstd = torch.rsqrt(var32 + eps)
    y32 = ((x32 - mean32[:, None]).to(F64) * (rstd[:, None] * d["gamma"]) + d["beta"].to(F64)).to(F32)
    offs = (mu.abs() / var.sqrt()).median().item()
    return ref, y32.to(out_dtype).to(F64), offs


# ------------------------------------------------------------------------------------------------------------------
# UP1 / UP2 (mask-decoder output up-scaling): GEMM columns n = (2 dy + dx) * C + c, pixel shuffle, skip, ...
# ------------------------------------------------------------------------------------------------------------------
def _shuffle(P, nb, gh, gw, C):
    """GEMM result [nb*gh*gw, 4*C] (columns (dy, dx, c)) -> [nb, 2gh, 2gw, C]: the ConvTranspose2d(k=2, s=2) output."""
    return P.view(nb, gh, gw, 2, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(nb, 2 * gh, 2 * gw, C)


def _skip_of(skip, bstride, prompts, gh, gw, C):
    if bstride == 0:
        return skip.view(1, 2 * gh, 2 * gw, C).expand(len(prompts), -1, -1, -1)
    return torch.stack([skip.view(-1)[p * bstride:p * bstride + 4 * gh * gw * C].view(2 * gh, 2 * gw, C) for p in prompts])


def up_inputs(stage, kind, B, gh, gw, per_prompt_skip, seed, device="cuda"):
    """UP1: keys [B*gh*gw, 256], w [256, 256]; UP2: u1 [B*gh*gw, 64], w [128, 64]. bias = a per-channel vector repeated
    over the 4 (dy, dx) groups, as ConvTranspose2d has it."""
    gen = torch.Generator(device=device).manual_seed(seed)
    K, C = (256, 64) if stage == 1 else (64, 32)
    a, w = _operands(kind, B * gh * gw, 4 * C, K, gen, device)
    d = dict(a=a.to(BF16), w=w.to(BF16), bias=(0.1 * torch.randn(C, generator=gen, device=device)).repeat(4).contiguous())
    nsk = B if per_prompt_skip else 1
    d["skip"] = torch.randn(nsk * 4 * gh * gw, C, generator=gen, device=device)
    d["bstride"] = 4 * gh * gw * C if per_prompt_skip else 0
    if stage == 1:
        d["gamma"] = 1.0 + 0.1 * torch.randn(C, generator=gen, device=device)
        d["beta"] = 0.1 * torch.randn(C, generator=gen, device=device)
    else:
        d["hyper"] = torch.randn(B, 4, C, generator=gen, device=device).contiguous()
    return d


def up_reference(stage, d, B, gh, gw, prompts, eps=1e-6):
    """(exact fp64, floor, envelope) of the listed prompts: UP1 -> [np, 2gh, 2gw, 64], UP2 -> [np, 4, 2gh, 2gw]."""
    C = 64 if stage == 1 else 32
    rows = torch.cat([torch.arange(p * gh * gw, (p + 1) * gh * gw, device=d["a"].device) for p in prompts])
    P = d["a"][rows].to(F64) @ d["w"].to(F64).t() + d["bias"].to(F64)
    x = _shuffle(P, len(prompts), gh, gw, C) + _skip_of(d["skip"], d["bstride"], prompts, gh, gw, C).to(F64)
    P32 = ((d["a"][rows].to(F64) @ d["w"].to(F64).t()).to(F32) + d["bias"])
    x32 = _shuffle(P32, len(prompts), gh, gw, C) + _skip_of(d["skip"], d["bstride"], prompts, gh, gw, C)
    if stage == 1:
        mu = x.mean(-1, keepdim=True)
        z = (x - mu) / torch.sqrt((x - mu).pow(2).mean(-1, keepdim=True) + eps) * d["gamma"].to(F64) + d["beta"].to(F64)
        mu32 = x32.mean(-1, keepdim=True)
        rstd = torch.rsqrt((x32 - mu32).pow(2).mean(-1, keepdim=True) + eps)
        z32 = ((x32 - mu32).to(F64) * (rstd * d["gamma"]) + d["beta"].to(F64)).to(F32)
        return _act_exact(z, ACT_GELU), _gelu_tanh_form(z32).to(BF16).to(F64), _gelu_env(z)
    h = d["hyper"][prompts].to(F64)  # [np, 4, 32]
    ref = torch.einsum("bmc,byxc->bmyx", h, _act_exact(x, ACT_GELU))
    floor = torch.einsum("bmc,byxc->bmyx", h, _gelu_tanh_form(x32).to(F64)).to(F32).to(F64)
    env = torch.einsum("bmc,byxc->bmyx", h.abs(), _gelu_env(x))
    return ref, floor, env


def _call_upscale(stage, d, B, gh, gw, out, plist=None):
    """sb_gemm_upscale1 / 2 on a caller-owned output buffer (ops.gemm_upscale* allocate theirs)."""
    from saber_b200 import lib
    L = lib.load()
    s = torch.cuda.current_stream().cuda_stream
    pl = (plist[0].data_ptr(), plist[1].data_ptr()) if plist else (None, None)
    if stage == 1:
        rc = L.sb_gemm_upscale1(d["a"].data_ptr(), d["a"].stride(0), d["w"].data_ptr(), d["w"].stride(0), B, gh, gw,
                                d["bias"].data_ptr(), d["skip"].data_ptr(), d["bstride"], d["gamma"].data_ptr(),
                                d["beta"].data_ptr(), 1e-6, out.data_ptr(), pl[0], pl[1], s)
    else:
        rc = L.sb_gemm_upscale2(d["a"].data_ptr(), d["a"].stride(0), d["w"].data_ptr(), d["w"].stride(0), B, gh, gw,
                                d["bias"].data_ptr(), d["skip"].data_ptr(), d["bstride"], d["hyper"].data_ptr(),
                                out.data_ptr(), pl[0], pl[1], s)
    lib.check(rc, f"sb_gemm_upscale{stage}")


def _up_view(stage, out, B, gh, gw):
    return out.view(B, 2 * gh, 2 * gw, 64) if stage == 1 else out


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ops():
    from saber_b200 import ops as _ops
    _ops.require_b200()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return _ops


@pytest.mark.gpu
@pytest.mark.parametrize("c", STD_CASES, ids=[c.id for c in STD_CASES])
def test_gemm_std(ops, c):
    for i, kind in enumerate(_kinds(c)):
        d = std_inputs(c, kind, seed=100 + i)
        out, buf = run_std(ops, c, d)
        case = f"{c.id} {kind}"
        assert_guard_intact(buf, c.M, c.N, case)
        ref, floor, env = std_reference(c, d)
        assert_close(out, ref, floor, case, fp32=c.out == F32, env=env)


@pytest.mark.gpu
@pytest.mark.parametrize("act,res_mod", [(ACT_GELU, None), (ACT_NONE, 1024)])
def test_gemm_fp32_validation(ops, act, res_mod):
    """Route: ops.gemm with fp32 weights (the fp32 validation mode: 6-term bf16 split product on the same kernel, K' =
    6 K, then the exact-erf GELU kernel). Reference: the fp64 product of the fp32 operands; fp32 bars."""
    M, N, K = 4225, 272, 200
    gen = torch.Generator(device="cuda").manual_seed(31)
    a, w = _operands("kbeacon", M, N, K, gen, "cuda")
    a, w = _guarded(a, 128, 24, F32, gen), _guarded(w, 64, 24, F32, gen)
    bias = 0.5 * torch.randn(N, generator=gen, device="cuda")
    res = _guarded(torch.randn(res_mod, N, generator=gen, device="cuda"), 32, 8, F32, gen) if res_mod else None
    # the exact-GELU pass runs over the output as one contiguous range: no extra columns there
    buf = _out_buffer(M, N, F32, "cuda", extra_cols=act != ACT_GELU)
    o = ops.gemm(a, w, bias, act, res, res_mod or 0, F32, out=buf[:M, :N])
    assert_guard_intact(buf, M, N, f"fp32 validation act{act}")
    x = a.to(F64) @ w.to(F64).t() + bias.to(F64)
    ref = _act_exact(x, act)
    floor = _act_exact(x.to(F32), act).to(F64)
    if res is not None:
        ref = ref + res[torch.arange(M, device="cuda") % res_mod].to(F64)
        floor = (floor.to(F32) + res[torch.arange(M, device="cuda") % res_mod]).to(F64)
    assert_close(o, ref, floor, f"fp32 validation act{act} res_mod{res_mod}", fp32=True)


LN_CASES = [(64, "f32"), (80, "bf16"), (128, "f32mod"), (256, "f32"), (256, "bf16"), (256, "f32mod"), (64, "bf16"),
            (80, "f32mod"), (128, "bf16"), (80, "f32"), (128, "f32"), (64, "f32mod")]


@pytest.mark.gpu
@pytest.mark.parametrize("N,res", LN_CASES)
def test_gemm_ln(ops, N, res):
    """Route: sb_gemm_ln (LayerNorm over the whole row in the epilogue; tile width 64 / 128 / 256 for N = 64, 80 and
    128, 256), residual fp32, bf16 or fp32 broadcast over res_mod rows, both output dtypes, with rows whose |mean| /
    std is 0, 64 and 256 (the residual stream of the mask decoder carries such rows into norm4)."""
    M, K = 4225, 200
    res_mod = 1024 if res == "f32mod" else 0
    for offset in (0, 64, 256):
        d = ln_inputs(M, N, K, "bf16" if res == "bf16" else "f32", res_mod, offset, seed=N + offset)
        for out_dtype in (BF16, F32):
            out = ops.gemm_ln(d["a"], d["w"], d["bias"], d["res"], d["gamma"], d["beta"], 1e-5, res_mod=res_mod,
                              out_dtype=out_dtype)
            ref, floor, offs = ln_reference(d, M, N, res_mod, 1e-5, out_dtype)
            assert_close(out, ref, floor, f"ln N{N} res {res} offset {offset} (|mean|/std {offs:.0f}) "
                         f"{'bf16' if out_dtype == BF16 else 'f32'}", fp32=out_dtype == F32)


UP_CASES = [(1, 16, 5, False), (1, 16, 5, True), (1, 64, 3, False), (1, 64, 3, True),
            (2, 16, 5, False), (2, 16, 5, True), (2, 64, 3, False), (2, 64, 3, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("stage,g,B,per_prompt", UP_CASES)
def test_gemm_upscale(ops, stage, g, B, per_prompt):
    """Routes: sb_gemm_upscale1 (ConvTranspose2d 256 -> 64 + feat_s1 + LayerNorm2d + GELU, bf16 out) and
    sb_gemm_upscale2 (ConvTranspose2d 64 -> 32 + feat_s0 + GELU, dot with the 4 hyper-network vectors, fp32 masks), on
    all prompts (ops.gemm_upscale*) and on a prompt list from ops.iou_gate written into a NaN-filled buffer: listed
    prompts within the bars, the other prompts' outputs untouched bit for bit."""
    gh = gw = g
    prompts = list(range(B))
    for kind in ("flat", "kbeacon"):
        d = up_inputs(stage, kind, B, gh, gw, per_prompt, seed=stage * 100 + g + B)
        if stage == 1:
            out = ops.gemm_upscale1(d["a"], d["w"], d["bias"], d["skip"], d["bstride"], d["gamma"], d["beta"], B, gh, gw)
        else:
            out = ops.gemm_upscale2(d["a"], d["w"], d["bias"], d["skip"], d["bstride"], d["hyper"], B, gh, gw)
        ref, floor, env = up_reference(stage, d, B, gh, gw, prompts)
        case = f"up{stage} {kind} gh{g} B{B} per_prompt_skip{per_prompt}"
        assert_close(_up_view(stage, out, B, gh, gw), ref, floor, case, fp32=stage == 2, env=env)
    # prompt list: prompts 1 and B - 1 pass the IoU gate
    listed = [1, B - 1]
    ious = torch.full((B, 4), 0.1, device="cuda")
    for p in listed:
        ious[p, 2] = 0.9
    plist = ops.iou_gate(ious, 0.5)
    assert plist[1].item() == len(listed) and plist[0][:len(listed)].tolist() == listed
    dt = BF16 if stage == 1 else F32
    shape = (B * 4 * gh * gw, 64) if stage == 1 else (B, 4, 2 * gh, 2 * gw)
    it = torch.int16 if dt == BF16 else torch.int32
    buf = torch.full(shape, NAN_BITS[dt], dtype=it, device="cuda").view(dt)
    _call_upscale(stage, d, B, gh, gw, buf, plist)
    torch.cuda.synchronize()
    view = _up_view(stage, buf, B, gh, gw)
    ref, floor, env = up_reference(stage, d, B, gh, gw, listed)
    assert_close(view[listed], ref, floor, f"{case} prompt list {listed}", fp32=stage == 2, env=env)
    others = [p for p in range(B) if p not in listed]
    bits = view[others].contiguous().view(it)
    assert (bits == NAN_BITS[dt]).all(), f"{case}: unlisted prompts {others} were written"


# ---- production shapes: every row of the bench step's GEMM list once, default route selection ---------------------
def _production_rows():
    rows = []
    with open(os.path.join(ROOT, "profiles", "r02zzzz_gemm_shapes.txt")) as f:
        for line in f:
            t = line.split()
            if not t:
                continue
            i = t.index("TFLOP/s")
            kind = t[i + 1]
            M, N, K = (int(t[i + 2 + j].split("=")[1]) for j in range(3))
            out = t[i + 5] if kind == "std" else None
            rows.append((kind, M, N, K, out, "+res" in t))
    return rows


PRODUCTION = _production_rows()


def _sample_rows(M, row_bytes, gen):
    """First / last 512 rows, 64 rows on each side of every 2^31-byte output offset, 4096 random rows."""
    s = set(range(min(M, 512))) | set(range(max(0, M - 512), M))
    for j in range(1, (M * row_bytes) // (1 << 31) + 1):
        r = (j << 31) // row_bytes
        s |= set(range(max(0, r - 64), min(M, r + 64)))
    s |= set(torch.randint(0, M, (4096,), generator=gen).tolist())
    return torch.tensor(sorted(s), dtype=torch.long)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,M,N,K,out,res", PRODUCTION,
                         ids=[f"{r[0]}-M{r[1]}-N{r[2]}-K{r[3]}{'-' + r[4] if r[4] else ''}{'-res' if r[5] else ''}"
                              for r in PRODUCTION])
def test_gemm_production_shapes(ops, kind, M, N, K, out, res):
    """Rows of profiles/r02zzzz_gemm_shapes.txt (a bench step's GEMMs) with the default route; the reference on a row
    sample (large products: outputs up to 2.4 GB, past the 2^31-byte offset)."""
    if kind in ("up1", "up2"):
        stage = 1 if kind == "up1" else 2
        g = 64 if stage == 1 else 128
        B = M // (g * g)
        d = up_inputs(stage, "flat", B, g, g, False, seed=M % 1000)
        if stage == 1:
            o = ops.gemm_upscale1(d["a"], d["w"], d["bias"], d["skip"], 0, d["gamma"], d["beta"], B, g, g)
        else:
            o = ops.gemm_upscale2(d["a"], d["w"], d["bias"], d["skip"], 0, d["hyper"], B, g, g)
        prompts = sorted({0, B // 2, B - 1})
        ref, floor, env = up_reference(stage, d, B, g, g, prompts)
        assert_close(_up_view(stage, o, B, g, g)[prompts], ref, floor, f"{kind} M{M}", fp32=stage == 2, env=env)
        return
    c = Std(M, N, K, 0, out, bias=True, res="f32" if res else None, route="default")
    gen = torch.Generator(device="cuda").manual_seed(M + N + K)
    a, w = _operands("flat", M, N, K, gen, "cuda")
    d = dict(a=a.to(BF16), w=w.to(BF16), bias=0.5 * torch.randn(N, generator=gen, device="cuda"), res=None)
    del a
    if res:
        d["res"] = torch.randn(M, N, generator=gen, device="cuda")
    o = ops.gemm(d["a"], d["w"], d["bias"], 0, d["res"], 0, c.out)
    rows = _sample_rows(M, N * (2 if c.out == BF16 else 4), torch.Generator().manual_seed(M)).cuda()
    ref, floor, _ = std_reference(c, d, rows=rows)
    assert_close(o[rows], ref, floor, f"production {c.id} ({rows.numel()} rows)", fp32=c.out == F32)


# ---- SM budget and single-CTA kernel in a child process (the environment is read once per process) ------------------
def _sm_cases():
    return [Std(70000, 272, 200, 0, "bf16", ACT_GELU, bias=True, route="default"),
            Std(40000, 576, 576, 0, "f32", bias=True, res="f32", route="default"),
            Std(20000, 1152, 288, 0, "bf16", bias=True, route="default"),
            Std(9000, 144, 1152, 0, "f32", bias=True, res="f32", res_mod=4096, route="default")]


def _sm_outputs(ops):
    outs = []
    for i, c in enumerate(_sm_cases()):
        d = std_inputs(c, "kbeacon", seed=300 + i)
        outs.append(run_std(ops, c, d)[0].clone())
    d = ln_inputs(20000, 256, 256, "bf16", 0, 0, seed=7)
    outs.append(ops.gemm_ln(d["a"], d["w"], d["bias"], d["res"], d["gamma"], d["beta"], 1e-5))
    d = up_inputs(1, "flat", 3, 64, 64, True, seed=8)
    outs.append(ops.gemm_upscale1(d["a"], d["w"], d["bias"], d["skip"], d["bstride"], d["gamma"], d["beta"], 3, 64, 64))
    return outs


@pytest.mark.gpu
def test_gemm_sm_budget_and_single_cta():
    """SB_GEMM_SMS=132 (persistent kernels on fewer CTAs) must give the default outputs bit for bit: every tile's
    accumulation and epilogue are the same whichever CTA runs it. SB_GEMM_2CTA=0 (every product on the single-CTA
    kernel) must be within the bars."""
    from saber_b200 import ops as _ops
    _ops.require_b200()
    default = [o.cpu() for o in _sm_outputs(_ops)]
    flags = ["-s"] if sys.flags.no_user_site else []
    with tempfile.TemporaryDirectory() as tmp:
        got = {}
        for name, extra in (("sms132", {"SB_GEMM_SMS": "132"}), ("single_cta", {"SB_GEMM_2CTA": "0"})):
            path = os.path.join(tmp, name + ".pt")
            env = dict(os.environ, **extra)
            r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), path], env=env, cwd=ROOT,
                               capture_output=True, text=True, timeout=900)
            assert r.returncode == 0, f"{name} child failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
            got[name] = torch.load(path)
    for i, (o, g) in enumerate(zip(default, got["sms132"])):
        assert torch.equal(_bits(o), _bits(g)), f"SB_GEMM_SMS=132 output {i} differs from the default"
    for i, c in enumerate(_sm_cases()):
        d = std_inputs(c, "kbeacon", seed=300 + i)
        ref, floor, env = std_reference(c, d)
        assert_close(got["single_cta"][i].cuda(), ref, floor, f"SB_GEMM_2CTA=0 {c.id}", fp32=c.out == F32, env=env)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the bars are attainable and catch the defects they exist for (float64 model, no kernel involved)
# ------------------------------------------------------------------------------------------------------------------
def _cpu_case(c):
    """The route's shape class at CPU size: at most 320 rows (res_mod kept when smaller)."""
    M = min(c.M, 320)
    return Std(M, c.N, c.K, c.bn, "bf16" if c.out == BF16 else "f32", c.act, c.bias, c.res,
               min(c.res_mod, 100 if c.res_mod % 32 else 64), c.alpha, c.route)


@pytest.mark.parametrize("c", STD_CASES, ids=[c.id for c in STD_CASES])
def test_cpu_std_floor_has_2x_margin(c):
    c = _cpu_case(c)
    for kind in _kinds(c):
        d = std_inputs(c, kind, seed=1, device="cpu")
        ref, floor, env = std_reference(c, d)
        bars = F32_BARS if c.out == F32 else BF16_BARS
        f = _errors(floor, ref, env)
        assert not _fails(f, tuple(None if b is None else b / 2 for b in bars)), (kind, f, bars)


@pytest.mark.parametrize("N,res", [(64, "f32"), (80, "bf16"), (256, "f32mod"), (256, "bf16")])
def test_cpu_ln_floor_has_2x_margin(N, res):
    res_mod = 32 if res == "f32mod" else 0
    for offset in (0, 64, 256):
        d = ln_inputs(256, N, 200, "bf16" if res == "bf16" else "f32", res_mod, offset, seed=2, device="cpu")
        for dt in (BF16, F32):
            ref, floor, _ = ln_reference(d, 256, N, res_mod, 1e-5, dt)
            bars = F32_BARS if dt == F32 else BF16_BARS
            f = _errors(floor, ref)
            assert not _fails(f, tuple(None if b is None else b / 2 for b in bars)), (offset, dt, f)


@pytest.mark.parametrize("stage", [1, 2])
def test_cpu_upscale_floor_and_layout(stage):
    """The floor has 2x margin, and the GEMM + pixel-shuffle form of the reference is ConvTranspose2d(k=2, s=2)."""
    import torch.nn.functional as F
    B, g = 2, 16
    d = up_inputs(stage, "flat", B, g, g, True, seed=3, device="cpu")
    ref, floor, env = up_reference(stage, d, B, g, g, [0, 1])
    bars = F32_BARS if stage == 2 else BF16_BARS
    f = _errors(floor, ref, env)
    assert not _fails(f, tuple(None if b is None else b / 2 for b in bars)), f
    C, K = (64, 256) if stage == 1 else (32, 64)
    wt = d["w"].to(F64).view(2, 2, C, K).permute(3, 2, 0, 1)  # [cin, cout, kh, kw]
    x = d["a"].to(F64).view(B, g, g, K).permute(0, 3, 1, 2)
    conv = F.conv_transpose2d(x, wt, d["bias"][:C].to(F64), stride=2).permute(0, 2, 3, 1)
    P = d["a"].to(F64) @ d["w"].to(F64).t() + d["bias"].to(F64)
    assert torch.allclose(_shuffle(P, B, g, g, C), conv, rtol=0, atol=1e-12)


def test_cpu_k_positions():
    assert k_positions(32) == [0, 31, 15, 16]
    assert k_positions(72) == [0, 71, 15, 16, 31, 32, 47, 48, 63, 64]
    p = k_positions(4608)
    assert {0, 4607, 63, 64, 575, 576, 4543, 4544} <= set(p) and len(p) == len(set(p))


# (defect, case, kinds on which it must fail a bar)
_DEFECT_CASES = [
    ("drop_kblock", Std(320, 272, 200, bias=True), ("flat", "kbeacon", "markers")),
    ("drop_kblock", Std(320, 272, 4608, out="f32", res="f32"), ("flat", "kbeacon", "markers")),
    ("drop_partial_tail", Std(320, 272, 200, bias=True), ("flat", "kbeacon", "markers")),
    ("drop_partial_tail", Std(320, 100, 72, act=ACT_GELU), ("flat", "kbeacon", "markers")),
    ("drop_partial_tail", Std(320, 32, 32), ("flat", "kbeacon", "markers")),
    ("row_moved_in_warp", Std(320, 272, 200, bias=True), ("flat", "kbeacon", "markers")),
    ("row_moved_in_warp", Std(320, 272, 4608, out="f32", res="f32"), ("flat", "kbeacon", "markers", "hotres")),
    ("residual_row_m", Std(320, 272, 200, res="bf16", res_mod=32), ("flat", "kbeacon", "markers", "hotres")),
    ("residual_row_m", Std(320, 4, 200, out="f32", res="f32", res_mod=100), ("flat", "kbeacon", "markers", "hotres")),
    ("bias_missing_last_tile", Std(320, 272, 200, bias=True), ("flat", "kbeacon", "markers")),
    ("bias_missing_last_tile", Std(320, 272, 72, out="f32", act=ACT_GELU, bias=True), ("flat", "kbeacon", "markers")),
    ("bf16_acc", Std(320, 272, 4608, out="f32", res="f32"), ("flat", "kbeacon", "markers")),
    ("bf16_acc", Std(320, 144, 200, out="f32", bias=True, res="f32", res_mod=64), ("flat", "kbeacon", "markers")),
    ("scale_0.998", Std(320, 272, 200, bias=True), ("flat", "kbeacon", "markers")),
    ("scale_0.998", Std(320, 272, 72, act=ACT_GELU, bias=True, res="bf16"), ("flat", "kbeacon", "markers", "hotres")),
    ("scale_0.998", Std(320, 272, 4608, out="f32", res="f32"), ("flat", "kbeacon", "markers", "hotres")),
]


@pytest.mark.parametrize("defect,c,kinds", _DEFECT_CASES,
                         ids=[f"{x[0]}-{x[1].id}" for x in _DEFECT_CASES])
def test_cpu_std_defect_fails_a_bar(defect, c, kinds):
    bars = F32_BARS if c.out == F32 else BF16_BARS
    for kind in kinds:
        d = std_inputs(c, kind, seed=5, device="cpu")
        ref, floor, env = std_reference(c, d, defect=defect)
        errs = _errors(floor, ref, env)
        assert _fails(errs, bars), f"{defect} passes the bars on {kind}: {errs}"


@pytest.mark.parametrize("N", [64, 256])
def test_cpu_ln_onepass_variance_fails_a_bar(N):
    """A one-pass fp32 variance of the raw values (sumsq / N - mean^2, what the LN epilogue computed before it summed
    x - x0) on rows with |mean| / std of 64 (fp32 output) and 256 (both outputs)."""
    for offset, dts in ((64, (F32,)), (256, (F32, BF16))):
        d = ln_inputs(256, N, 200, "f32", 0, offset, seed=4, device="cpu")
        for dt in dts:
            ref, floor, _ = ln_reference(d, 256, N, 0, 1e-5, dt, defect="onepass_variance")
            errs = _errors(floor, ref)
            assert _fails(errs, F32_BARS if dt == F32 else BF16_BARS), (offset, dt, errs)


if __name__ == "__main__":  # child of test_gemm_sm_budget_and_single_cta: write the outputs under this environment
    sys.path.insert(0, ROOT)
    from saber_b200 import ops as _child_ops
    _child_ops.require_b200()
    torch.save([o.cpu() for o in _sm_outputs(_child_ops)], sys.argv[1])
