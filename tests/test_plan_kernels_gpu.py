"""Element-wise tests of the launches the UNet / VAE / CLIP plans build, through the plans' own builders.

The sdxl_op_* entry points (test_ops_gpu.py) build their own simple launches. What the plans launch is recorded by PlanBuilder
(csrc/engine_core.h) with weights re-laid out by the Loader: fused skip segments, per-image bias rows, phase-decomposed upsample
convs, the hi/lo-split head, column windows of fused QKV / KV matrices, the VAE's single-head attention and PaddedConv2d. The
sdxl_dbg_plan_* entry points run exactly that code on test data; every reference here is float64 (torch on the GPU) on the
same f16 operands the kernel reads.

Tolerances:
- GEMM-shaped ops, every output element: |out - ref| <= K_eff * 2^-23 * (|a| * |w| + |bias| + |res|), the worst-case error of
  f32 accumulation, with K_eff = Ktot / 8 + 4 (one rounding per 16-deep tensor-core step, counted twice for the alignment of
  the products inside a step, plus bias and residual). An f16 output adds 2^-11 |ref|. A correct kernel cannot fail this; a
  missing or duplicated tap, another image's bias, a phase written to the wrong pixel or a head reading the wrong columns does.
  Relative L2 <= 1e-5 * max(1, sqrt(Ktot / 2880)) for f32 outputs: test_ops_gpu.py's 1e-5 up to its largest K (2880); the
  accumulation error grows with K (measured on a B200: 3.4e-6 at K = 2880, 9.3e-6 at 11520, 1.27e-5 at 14080). Worst
  element ratio measured: 0.05 for f32 outputs, 0.94 for f16 outputs (their output rounding is most of the bound).
- The output head is compared with the f64 conv of the *unrounded* normalised activation (f64 GroupNorm + SiLU): the hi/lo
  split must make it f32-exact: relative L2 <= 1e-5 and at least 10x below the error of the f16 activation alone (measured:
  8.7e-6 against 2.1e-4 at 128^2, 7.9e-6 against 1.8e-4 at 16^2).
- GroupNorm: y + y_lo within 1e-5 absolute of the f64 GroupNorm on O(1) data (measured max 1.2e-6; y alone 1.9e-3) and at
  least 20x closer than y alone; raw == f16(cat(x1, x2)) bitwise.
- Attention (f16 output): relative L2 <= 1e-3 against f64 softmax(q k^T / sqrt(d)) v (measured max 3.4e-4), and per (query
  row, head) relative error <= ATTN_ROW_TOL, about twice the largest value measured on a B200 (1000 W power limit) over the
  cases below: tensor-core kernel 5.2e-4, short-sequence kernel 3.0e-4, VAE single-head core (per row and 64-column block)
  4.9e-4. The VAE core's softmax_rows is checked on the kernel's own scores (f32 math, one f16 rounding per probability)
  and transpose_f16 bitwise.
- Outputs carry NaN sentinels (extra rows, ldo > N): nothing outside the logical output may change.
- Each GEMM case declares the implicit-GEMM variant it covers; the test asserts the launch ran it, and
  test_variant_coverage asserts that the declared variants cover every one the default heuristic can produce. The A/B switches
  (SDXL_B200_PAIR / _CLUSTER / _EPI_TMA / _EPI_COMPACT, read once per process) are run in a subprocess each.
"""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from sdxl_b200 import _lib
from sdxl_b200.weights import build_pack

pytestmark = pytest.mark.gpu

U = 2.0 ** -23
H16 = 2.0 ** -11
ATTN_ROW_TOL = {"flash": 1.1e-3, "small": 6e-4, "vae": 1e-3}
FIELDS = ("pair", "CM", "CN", "split", "BN", "nstages", "epi_tma", "box")
CONV3, UPCONV, HEAD, PADDED, LINEAR, LINEAR_F16, GEGLU = range(7)
# set in the subprocesses of test_ab_switch: the forced setting replaces the declared variants
FORCED = os.environ.get("SDXL_B200_PLAN_TEST_FORCED", "")


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def randn(g, *shape, scale=1.0):
    return torch.randn(*shape, device="cuda", generator=g) * scale


def f16r(t):
    """values exactly representable in f16, as f32"""
    return t.half().float()


def pack(tensors):
    return build_pack({k: v.detach().cpu().half().contiguous() for k, v in tensors.items()}, device="cpu").numpy().tobytes()


def ptr(t):
    return None if t is None else t.data_ptr()


def nan_buf(rows, cols, dtype):
    return torch.full((rows, cols), float("nan"), device="cuda", dtype=dtype)


def check_sentinel(buf, rows, cols, name):
    keep = torch.ones_like(buf, dtype=torch.bool)
    keep[:rows, :cols] = False
    assert torch.isnan(buf[keep].float()).all(), f"{name}: write outside the logical [{rows}, {cols}] output"


def check_bound(name, out, ref, absref, keff, f16_out=False):
    """element-wise worst-case bound; returns the worst normalised error"""
    err = (out.double() - ref).abs()
    bound = keff * U * absref + (H16 * ref.abs() if f16_out else 0.0) + 1e-30
    worst = float((err / bound).max())
    rel = float((out.double() - ref).norm() / ref.norm())
    print(f"  {name}: worst |err|/bound {worst:.3f}, rel L2 {rel:.2e}")
    assert torch.isfinite(out).all(), f"{name}: non-finite output"
    assert worst <= 1.0, f"{name}: element error above the f32 accumulation bound (worst ratio {worst:.2f})"
    return worst, rel


def run_gemm(kind, tensors, B, H, W, Cin, Cout, C2=0, x=None, x2=None, bias_rows=None, bias_ld=0, bias_off=0, res=None,
             out=None, ldo=0, ctx=None):
    lib = _lib.load()
    pk = pack(tensors)
    cfg = (C.c_int32 * (16 * len(FIELDS)))()
    ctx.enter()
    rc = lib.sdxl_dbg_plan_gemm(ctx.h, kind, pk, len(pk), B, H, W, Cin, Cout, C2, ptr(x), ptr(x2), ptr(bias_rows), bias_ld,
                                bias_off, ptr(res), ptr(out), ldo, cfg, 16)
    ctx.check(rc, "sdxl_dbg_plan_gemm")
    ctx.leave()
    rows = [tuple(cfg[i * 8:(i + 1) * 8]) for i in range(16)]
    return [dict(zip(FIELDS, r)) for r in rows if r[0] != -1]


def check_variant(name, cfgs, want):
    print("  PLANCFG " + json.dumps({"case": name, "cfg": cfgs}))
    if FORCED:
        return
    for c in cfgs:
        for k, v in want.items():
            assert c[k] == v, f"{name}: expected {k}={v}, the launch ran {c}"


def rel_tol(ktot):
    return 1e-5 * max(1.0, math.sqrt(ktot / 2880))


def conv_abs(x, w, **kw):
    return F.conv2d(x.abs(), w.abs(), **kw)


# ---------------------------------------------------------------------------------------------------------------------------
# variants: split 0/1/2 = A tile sliced along W/H/B across the CN peers; box 4096 = f32 boxes, 2048 = compact f16 boxes
V_PAIR = {"pair": 1, "CM": 2, "CN": 1}
V_1x1 = {"pair": 0, "CM": 1, "CN": 1}
V_2x1 = {"pair": 0, "CM": 2, "CN": 1}
V_1x2 = {"pair": 0, "CM": 1, "CN": 2}
V_2x2 = {"pair": 0, "CM": 2, "CN": 2}
TMA = {"epi_tma": 1}
STG = {"epi_tma": 0}

# name, B, H, W, Cin, Cout, C2 (skip), per-image bias, residual, declared variant
CONV3_CASES = [
    ("128x128 320", 1, 128, 128, 320, 320, 0, False, False, {**V_PAIR, **TMA}),
    ("64x64 640 res", 2, 64, 64, 640, 640, 0, False, True, {**V_PAIR, **TMA}),
    ("32x32 1280 temb", 2, 32, 32, 1280, 1280, 0, True, False, {**V_PAIR, **TMA}),
    ("32x32 skip 1280+1280", 1, 32, 32, 1280, 1280, 2560, False, False, {**V_PAIR, **TMA}),
    ("64x64 skip 640+320", 1, 64, 64, 640, 640, 960, False, False, {**V_PAIR, **TMA}),
    ("128x128 skip 320+320", 1, 128, 128, 320, 320, 640, False, False, {**V_PAIR, **TMA}),
    ("8x8 B3 temb", 3, 8, 8, 640, 640, 0, True, True, {**V_PAIR, **TMA}),
    ("4x4 B3 temb", 3, 4, 4, 1280, 1280, 0, True, False, {**V_1x2, "split": 2, **TMA}),
    ("2x2 B5 temb", 5, 2, 2, 1280, 1280, 0, True, True, {**V_1x2, "split": 2, **TMA}),
    ("4x4 B5 temb 128->80", 5, 4, 4, 128, 80, 0, True, True, {**V_1x1, **STG}),
    ("2x2 B5 temb 64->48", 5, 2, 2, 64, 48, 0, True, False, {**V_1x1, **STG}),
    ("12x20 72->48 temb res", 2, 12, 20, 72, 48, 0, True, True, {**V_2x1, **STG}),
    ("20x24 136->80 skip 200", 1, 20, 24, 136, 80, 200, False, False, {**V_1x1, **STG}),
    ("24x16 320 split H", 1, 24, 16, 320, 320, 0, False, True, {**V_1x2, "split": 1, **TMA}),
]


@pytest.mark.parametrize("case", CONV3_CASES, ids=[c[0] for c in CONV3_CASES])
def test_conv3(ctx, case):
    name, B, H, W, Cin, Cout, C2, temb, with_res, want = case
    g = gen(B * 1000 + H * 10 + Cin + C2)
    x = randn(g, B, H, W, Cin).half()
    x2 = randn(g, B, H, W, C2).half() if C2 else None
    w = f16r(randn(g, Cout, Cin, 3, 3, scale=1 / math.sqrt(9 * Cin)))
    b = f16r(randn(g, Cout, scale=0.1))
    t = {"conv/weight": w, "conv/bias": b}
    if C2:
        ws = f16r(randn(g, Cout, C2, 1, 1, scale=1 / math.sqrt(C2)))
        bs = f16r(randn(g, Cout, scale=0.1))
        t.update({"skip/weight": ws, "skip/bias": bs})
    ld, off = 3 * Cout + 16, Cout + 8
    bias_rows = randn(g, B, ld) if temb else None
    res = randn(g, B * H * W, Cout) if with_res else None
    extra = 37
    out = nan_buf(B * H * W + extra, Cout, torch.float32)
    cfgs = run_gemm(CONV3, t, B, H, W, Cin, Cout, C2, x, x2, bias_rows, ld, off, res, out, Cout, ctx=ctx)
    xn = x.double().permute(0, 3, 1, 2)
    wd = w.double()
    ref = F.conv2d(xn, wd, padding=1)
    absref = conv_abs(xn, wd, padding=1)
    if C2:
        x2n = x2.double().permute(0, 3, 1, 2)
        ref = ref + F.conv2d(x2n, ws.double())
        absref = absref + conv_abs(x2n, ws.double())
    if temb:
        bias = bias_rows.double()[:, off:off + Cout]                       # one bias row per image
    else:
        bias = (b.double() + (bs.double() if C2 else 0.0)).expand(B, Cout)
    ref = ref + bias[:, :, None, None]
    absref = absref + bias.abs()[:, :, None, None]
    ref = ref.permute(0, 2, 3, 1).reshape(B * H * W, Cout)
    absref = absref.permute(0, 2, 3, 1).reshape(B * H * W, Cout)
    if with_res:
        ref = ref + res.double()
        absref = absref + res.double().abs()
    Ktot = 9 * ((Cin + 63) // 64 * 64) + (C2 + 63) // 64 * 64
    _, rel = check_bound(name, out[:B * H * W], ref, absref, Ktot / 8 + 4)
    assert rel <= rel_tol(Ktot)
    check_sentinel(out, B * H * W, Cout, name)
    check_variant(name, cfgs, want)


def upconv_phase_weights(w):
    """The rule of repack_upconv_launch (csrc/kernels.h): a 3x3 conv on the nearest-2x upsampled image is, for output parity
    (a, b), a 2x2 conv on the source image; the 3x3 taps that read the same source pixel are summed in f32 and rounded once to
    f16. Row parity a = 0 reads source rows i-1 (tap 0) and i (taps 1, 2); a = 1 reads rows i (taps 0, 1) and i+1 (tap 2);
    columns likewise. Returns {(a, b): [O, I, 2, 2]} as float64 values of f16 numbers."""
    groups = {0: [[0], [1, 2]], 1: [[0, 1], [2]]}
    out = {}
    for a in (0, 1):
        for b in (0, 1):
            k = torch.zeros(w.shape[0], w.shape[1], 2, 2, dtype=torch.float32, device=w.device)
            for th, khs in enumerate(groups[a]):
                for tw, kws in enumerate(groups[b]):
                    for kh in khs:
                        for kw in kws:
                            k[:, :, th, tw] += w[:, :, kh, kw].float()
            out[(a, b)] = k.half().double()
    return out


UPCONV_CASES = [
    ("4x4 B3 1280", 3, 4, 4, 1280, {**V_1x2, **STG}),
    ("8x8 B2 1280", 2, 8, 8, 1280, {**V_1x2, "split": 2, **STG}),
    ("12x20 1280", 1, 12, 20, 1280, {**V_PAIR, **STG}),
    ("32x32 1280", 1, 32, 32, 1280, {**V_PAIR, **STG}),
    ("64x64 640", 1, 64, 64, 640, {**V_PAIR, **STG}),
]


@pytest.mark.parametrize("case", UPCONV_CASES, ids=[c[0] for c in UPCONV_CASES])
def test_upconv(ctx, case):
    name, B, H, W, Cc, want = case
    g = gen(B * 77 + H * 5 + W + Cc)
    x = f16r(randn(g, B, H, W, Cc))
    w = f16r(randn(g, Cc, Cc, 3, 3, scale=1 / math.sqrt(9 * Cc)))
    b = f16r(randn(g, Cc, scale=0.1))
    rows = B * 4 * H * W
    out = nan_buf(rows + 29, Cc, torch.float32)
    cfgs = run_gemm(UPCONV, {"conv/weight": w, "conv/bias": b}, B, H, W, Cc, Cc, x=x, out=out, ldo=Cc, ctx=ctx)
    assert len(cfgs) == 4
    xn = F.pad(x.double().permute(0, 3, 1, 2), (1, 1, 1, 1))
    ph = upconv_phase_weights(w)
    ref = torch.empty(B, Cc, 2 * H, 2 * W, dtype=torch.float64, device="cuda")
    absref = torch.empty_like(ref)
    for (a, bb), k in ph.items():
        xs = xn[:, :, a:a + H + 1, bb:bb + W + 1]
        ref[:, :, a::2, bb::2] = F.conv2d(xs, k) + b.double()[None, :, None, None]
        absref[:, :, a::2, bb::2] = conv_abs(xs, k) + b.double().abs()[None, :, None, None]
    o = out[:rows].reshape(B, 2 * H, 2 * W, Cc).permute(0, 3, 1, 2)
    _, rel = check_bound(name, o, ref, absref, 4 * ((Cc + 63) // 64 * 64) / 8 + 4)
    assert rel <= 1e-5
    # the phase decomposition against the layer it replaces: nearest-2x upsample, then the 3x3 conv with the f16 weights
    true = F.conv2d(F.interpolate(x.double().permute(0, 3, 1, 2), scale_factor=2, mode="nearest"), w.double(), b.double(), padding=1)
    rel_true = float((o.double() - true).norm() / true.norm())
    print(f"  {name}: rel L2 against interpolate + conv2d {rel_true:.2e}")
    assert rel_true <= 1e-3
    check_sentinel(out, rows, Cc, name)
    check_variant(name, cfgs, want)


def gn64(x, gamma, beta, silu, eps=1e-5):
    B, HW, Cc = x.shape
    xg = x.double().reshape(B, HW, 32, Cc // 32)
    mean = xg.mean(dim=(1, 3), keepdim=True)
    var = ((xg - mean) ** 2).mean(dim=(1, 3), keepdim=True)
    t = ((xg - mean) / torch.sqrt(var + eps)).reshape(B, HW, Cc) * gamma.double() + beta.double()
    return t * torch.sigmoid(t) if silu else t


HEAD_CASES = [("128x128 B2 320->4", 2, 128, 128, 320, {**V_2x1, **STG}), ("16x16 320->4", 1, 16, 16, 320, STG)]


@pytest.mark.parametrize("case", HEAD_CASES, ids=[c[0] for c in HEAD_CASES])
def test_head_hilo(ctx, case):
    name, B, H, W, Cc, want = case
    g = gen(H + Cc + B)
    x = randn(g, B, H, W, Cc, scale=1.5) + 0.3
    gamma, beta = f16r(1 + randn(g, Cc, scale=0.2)), f16r(randn(g, Cc, scale=0.2))
    w = f16r(randn(g, 4, Cc, 3, 3, scale=1 / math.sqrt(9 * Cc)))
    b = f16r(randn(g, 4, scale=0.1))
    t = {"norm/weight": gamma, "norm/bias": beta, "conv/weight": w, "conv/bias": b}
    rows = B * H * W
    ldo = 8
    out = nan_buf(rows + 19, ldo, torch.float32)
    cfgs = run_gemm(HEAD, t, B, H, W, Cc, 4, x=x, out=out, ldo=ldo, ctx=ctx)
    act = gn64(x.reshape(B, H * W, Cc), gamma, beta, True).reshape(B, H, W, Cc).permute(0, 3, 1, 2)
    ref = F.conv2d(act, w.double(), b.double(), padding=1).permute(0, 2, 3, 1).reshape(rows, 4)
    absref = (conv_abs(act, w.double(), padding=1) + b.double().abs()[None, :, None, None]).permute(0, 2, 3, 1).reshape(rows, 4)
    # K = [9 taps on hi | 9 taps on lo]
    _, rel = check_bound(name, out[:rows, :4], ref, absref, 2 * 9 * ((Cc + 63) // 64 * 64) / 8 + 4)
    # what the f16 activation alone would give: the same conv on y = f16(t)
    y = act.half().double()
    rel_hi = float((F.conv2d(y, w.double(), b.double(), padding=1).permute(0, 2, 3, 1).reshape(rows, 4) - ref).norm() / ref.norm())
    print(f"  {name}: rel L2 {rel:.2e} against the unrounded activation; f16 activation alone {rel_hi:.2e}")
    assert rel <= rel_tol(2 * 9 * 320) and rel * 10 <= rel_hi
    check_sentinel(out, rows, 4, name)
    check_variant(name, cfgs, want)


PADDED_CASES = [("8x8 B2 512", 2, 8, 8, 512, {**V_1x2, "split": 2, **TMA}), ("16x24 256", 1, 16, 24, 256, {**V_PAIR, **STG}),
                ("64x64 128", 1, 64, 64, 128, {**V_PAIR, **TMA})]


@pytest.mark.parametrize("case", PADDED_CASES, ids=[c[0] for c in PADDED_CASES])
def test_padded_conv_s2(ctx, case):
    name, B, H, W, Cc, want = case
    g = gen(B + H * 3 + W + Cc)
    x = f16r(randn(g, B, H, W, Cc))
    w = f16r(randn(g, Cc, Cc, 3, 3, scale=1 / math.sqrt(9 * Cc)))
    b = f16r(randn(g, Cc, scale=0.1))
    rows = B * (H // 2) * (W // 2)
    out = nan_buf(rows + 23, Cc, torch.float32)
    cfgs = run_gemm(PADDED, {"conv/weight": w, "conv/bias": b}, B, H, W, Cc, Cc, x=x, out=out, ldo=Cc, ctx=ctx)
    xp = F.pad(x.double().permute(0, 3, 1, 2), (0, 1, 0, 1))   # PaddedConv2d: zeros past the right and bottom edges only
    ref = F.conv2d(xp, w.double(), b.double(), stride=2).permute(0, 2, 3, 1).reshape(rows, Cc)
    absref = (conv_abs(xp, w.double(), stride=2) + b.double().abs()[None, :, None, None]).permute(0, 2, 3, 1).reshape(rows, Cc)
    _, rel = check_bound(name, out[:rows], ref, absref, 9 * Cc / 8 + 4)
    assert rel <= 1e-5
    check_sentinel(out, rows, Cc, name)
    check_variant(name, cfgs, want)


# name, kind, M, K, N, residual, ldo pad, declared variant
LINEAR_CASES = [
    ("4096x640x640 res", LINEAR, 4096, 640, 640, True, 32, {**V_PAIR, **TMA, "box": 4096}),
    ("1024x320x300", LINEAR, 1024, 320, 300, False, 4, {**V_2x2, "split": 0, **STG}),
    ("154x2048x1280", LINEAR, 154, 2048, 1280, False, 64, {**V_PAIR, **TMA}),
    ("200x136x48 res", LINEAR, 200, 136, 48, True, 16, {**V_1x1, **STG}),
    ("384x640x640 res", LINEAR, 384, 640, 640, True, 0, {**V_1x2, "split": 0, **TMA}),
    ("4096x640x1920 f16", LINEAR_F16, 4096, 640, 1920, False, 64, {**V_PAIR, **TMA, "box": 2048}),
    ("300x320x320 f16", LINEAR_F16, 300, 320, 320, False, 32, {**V_1x2, "split": 0, "epi_tma": 1, "box": 2048}),
    ("1024x640 geglu", GEGLU, 1024, 640, 5120, False, 64, {**V_PAIR, "epi_tma": 1, "box": 2048}),
    ("130x320 geglu", GEGLU, 130, 320, 2560, False, 0, {**V_PAIR, "epi_tma": 1, "box": 2048}),
]


@pytest.mark.parametrize("case", LINEAR_CASES, ids=[c[0] for c in LINEAR_CASES])
def test_linear(ctx, case):
    name, kind, M, K, N, with_res, pad, want = case
    g = gen(M + K * 3 + N * 7)
    x = randn(g, M, K).half()
    w = f16r(randn(g, K, N, scale=1 / math.sqrt(K)))
    b = f16r(randn(g, N, scale=0.1))
    n_out = N // 2 if kind == GEGLU else N
    ldo = n_out + pad
    f16_out = kind != LINEAR
    out = nan_buf(M + 41, ldo, torch.float16 if f16_out else torch.float32)
    res = randn(g, M, ldo) if with_res else None
    cfgs = run_gemm(kind, {"lin/weight": w, "lin/bias": b}, 1, 1, M, K, N, x=x, res=res, out=out, ldo=ldo, ctx=ctx)
    keff = ((K + 63) // 64 * 64) / 8 + 4
    h = x.double() @ w.double() + b.double()
    habs = x.double().abs() @ w.double().abs() + b.double().abs()
    if kind == GEGLU:
        # out = h[:, :n] * gelu_erf(h[:, n:]): the bound of each factor, through |d(a*gelu(g))| <= |gelu(g)||da| + 1.13|a||dg|
        a, gt = h[:, :n_out], h[:, n_out:]
        ref = a * F.gelu(gt)
        err_bound = keff * U * (F.gelu(gt).abs() * habs[:, :n_out] + 1.13 * a.abs() * habs[:, n_out:]) + 1e-6 * ref.abs()
        o = out[:M, :n_out].double()
        worst = float(((o - ref).abs() / (err_bound + H16 * ref.abs() + 1e-30)).max())
        rel = float((o - ref).norm() / ref.norm())
        print(f"  {name}: worst |err|/bound {worst:.3f}, rel L2 {rel:.2e}")
        assert worst <= 1.0 and rel <= 1e-3
    else:
        ref, absref = h, habs
        if with_res:
            ref = ref + res[:, :N].double()
            absref = absref + res[:, :N].double().abs()
        _, rel = check_bound(name, out[:M, :N], ref, absref, keff, f16_out=f16_out)
        assert rel <= (1e-3 if f16_out else 1e-5)
    check_sentinel(out, M, n_out, name)
    check_variant(name, cfgs, want)


def test_variant_coverage():
    """The declared variants of the GEMM cases cover every variant the default heuristic produces."""
    cases = [c[-1] for c in CONV3_CASES + UPCONV_CASES + HEAD_CASES + PADDED_CASES + LINEAR_CASES]
    have = lambda **kv: any(all(c.get(k) == v for k, v in kv.items()) for c in cases)  # noqa: E731
    assert have(pair=1) and have(pair=0)
    for cm, cn in ((1, 1), (1, 2), (2, 1), (2, 2)):
        assert have(pair=0, CM=cm, CN=cn), f"cluster {cm}x{cn} not covered"
    for split in (0, 1, 2):
        assert have(CN=2, split=split), f"A split along {'WHB'[split]} not covered"
    assert have(epi_tma=1) and have(epi_tma=0)
    assert have(epi_tma=1, box=4096) and have(epi_tma=1, box=2048)
    geglu = [c[-1] for c in LINEAR_CASES if c[1] == GEGLU]
    assert any(c.get("epi_tma") == 1 for c in geglu)


# ---------------------------------------------------------------------------------------------------------------------------
def test_group_norm_outputs(ctx):
    lib = _lib.load()
    for B, HW, C1, C2, silu in [(2, 1024, 320, 0, 1), (1, 4096, 640, 320, 1), (2, 256, 1280, 0, 0), (3, 64, 64, 64, 1)]:
        g = gen(HW + C1 + C2)
        x1 = randn(g, B, HW, C1, scale=1.5) + 0.3
        x2 = (randn(g, B, HW, C2, scale=0.7) - 0.2) if C2 else None
        Ct = C1 + C2
        gamma, beta = f16r(1 + randn(g, Ct, scale=0.2)), f16r(randn(g, Ct, scale=0.2))
        pk = pack({"norm/weight": gamma, "norm/bias": beta})
        y, raw, ylo = (torch.full((B, HW, Ct), float("nan"), device="cuda", dtype=torch.float16) for _ in range(3))
        ctx.enter()
        ctx.check(lib.sdxl_dbg_plan_group_norm(ctx.h, pk, len(pk), ptr(x1), C1, ptr(x2), C2, B, HW, silu, ptr(y), ptr(raw), ptr(ylo)),
                  "sdxl_dbg_plan_group_norm")
        ctx.leave()
        xc = torch.cat([x1, x2], dim=2) if C2 else x1
        ref = gn64(xc, gamma, beta, silu)
        e_hilo = float((y.double() + ylo.double() - ref).abs().max())
        e_hi = float((y.double() - ref).abs().max())
        print(f"  GN B={B} HW={HW} C={C1}+{C2} silu={silu}: |y + y_lo - ref| max {e_hilo:.2e}, |y - ref| max {e_hi:.2e}")
        assert torch.equal(raw, xc.half())
        assert e_hilo <= 1e-5 and e_hilo * 20 <= e_hi


# ---------------------------------------------------------------------------------------------------------------------------
def attn64(q, k, v, n_head, mask=None, causal=False):
    """q [B,T,C], k/v [B,S,C] -> f64 softmax(q k^T / 8) v per head"""
    B, T, Cc = q.shape
    S = k.shape[1]
    qh = q.double().reshape(B, T, n_head, 64).transpose(1, 2)
    kh = k.double().reshape(B, S, n_head, 64).transpose(1, 2)
    vh = v.double().reshape(B, S, n_head, 64).transpose(1, 2)
    s = qh @ kh.transpose(-1, -2) / 8.0
    if mask is not None:
        s = s + mask.double()
    if causal:
        s = s.masked_fill(torch.ones(T, S, device=s.device, dtype=torch.bool).triu(1), float("-inf"))
    return (torch.softmax(s, dim=-1) @ vh).transpose(1, 2).reshape(B, T, Cc)


def check_attn(name, out, ref, n_head, row_tol):
    B, T, Cc = ref.shape
    o = out.double()
    rel = float((o - ref).norm() / ref.norm())
    d = (o - ref).reshape(B, T, n_head, 64).norm(dim=-1)
    r = ref.reshape(B, T, n_head, 64).norm(dim=-1)
    row = float((d / r).max())
    print(f"  {name}: rel L2 {rel:.2e}, worst (row, head) rel {row:.2e}")
    assert torch.isfinite(o).all() and rel <= 1e-3 and row <= row_tol


def run_attn(ctx, small, q, qp, qc, kv, kvp, kc, vc, B, T, S, nh, out, ldo, mask=None, causal=0):
    lib = _lib.load()
    ctx.enter()
    ctx.check(lib.sdxl_dbg_plan_attention(ctx.h, small, ptr(q), qp, qc, ptr(kv), kvp, kc, vc, B, T, S, nh, ptr(mask), causal,
                                          ptr(out), ldo), "sdxl_dbg_plan_attention")
    ctx.leave()


# name, B, T, S (None: self-attention on a fused [M, 3C] QKV matrix), n_head
ATTN_CASES = [("self 5 heads T4096", 1, 4096, None, 5), ("self 10 heads B2 T1024", 2, 1024, None, 10),
              ("self 20 heads B2 T256", 2, 256, None, 20), ("cross 10 heads B2 T1024 S77", 2, 1024, 77, 10),
              ("cross 20 heads B2 T200 S333", 2, 200, 333, 20), ("self 2 heads T4096", 1, 4096, None, 2)]


@pytest.mark.parametrize("case", ATTN_CASES, ids=[c[0] for c in ATTN_CASES])
def test_attention_windows(ctx, case):
    name, B, T, S, nh = case
    Cc = nh * 64
    g = gen(B * T + nh)
    ldo = Cc + 64
    out = torch.full((B * T + 17, ldo), float("nan"), device="cuda", dtype=torch.float16)
    if S is None:    # q | k | v = columns [0, C) | [C, 2C) | [2C, 3C) of one [B*T, 3C] matrix, as the self-attention plan
        qkv = randn(g, B * T, 3 * Cc).half()
        run_attn(ctx, 0, qkv, 3 * Cc, 0, qkv, 3 * Cc, Cc, 2 * Cc, B, T, T, nh, out, ldo)
        q, k, v = (qkv[:, i * Cc:(i + 1) * Cc].reshape(B, T, Cc) for i in range(3))
    else:            # cross-attention: q [B*T, C], k | v = columns of one [B*S, 2C] matrix
        q2 = randn(g, B * T, Cc).half()
        kv = randn(g, B * S, 2 * Cc).half()
        run_attn(ctx, 0, q2, Cc, 0, kv, 2 * Cc, 0, Cc, B, T, S, nh, out, ldo)
        q = q2.reshape(B, T, Cc)
        k, v = kv[:, :Cc].reshape(B, S, Cc), kv[:, Cc:].reshape(B, S, Cc)
    check_attn(name, out[:B * T, :Cc].reshape(B, T, Cc), attn64(q, k, v, nh), nh, ATTN_ROW_TOL["flash"])
    check_sentinel(out, B * T, Cc, name)


@pytest.mark.parametrize("B,nh,causal", [(1, 12, 1), (4, 12, 0), (2, 20, 1), (3, 20, 0)])
def test_attention_small(ctx, B, nh, causal):
    """The text encoders' attention: fused QKV windows of pitch 3C, causal flag or an additive [T,S] mask."""
    T = 77
    Cc = nh * 64
    g = gen(B * 31 + nh + causal)
    qkv = randn(g, B * T, 3 * Cc).half()
    mask = None
    if not causal:
        mask = torch.where(torch.rand(T, T, device="cuda", generator=g) < 0.3, -1e4, 0.0)
        mask.fill_diagonal_(0.0)
        mask = (mask + randn(g, T, T, scale=0.5)).half()
    ldo = Cc + 32
    out = torch.full((B * T + 5, ldo), float("nan"), device="cuda", dtype=torch.float16)
    run_attn(ctx, 1, qkv, 3 * Cc, 0, qkv, 3 * Cc, Cc, 2 * Cc, B, T, T, nh, out, ldo, mask=mask, causal=causal)
    q, k, v = (qkv[:, i * Cc:(i + 1) * Cc].reshape(B, T, Cc) for i in range(3))
    name = f"attention_small B={B} heads={nh} {'causal' if causal else 'mask'}"
    check_attn(name, out[:B * T, :Cc].reshape(B, T, Cc), attn64(q, k, v, nh, mask, bool(causal)), nh, ATTN_ROW_TOL["small"])
    check_sentinel(out, B * T, Cc, name)


@pytest.mark.parametrize("T", [64, 192, 1024, 4096, 16384])
def test_vae_attention_core(ctx, T):
    lib = _lib.load()
    Cc = 512
    g = gen(T)
    q, k, v = (randn(g, T, Cc, scale=0.5).half() for _ in range(3))
    S = torch.full((T, T), float("nan"), device="cuda")
    Pm = torch.full((T, T), float("nan"), device="cuda", dtype=torch.float16)
    vT = torch.full((Cc, T), float("nan"), device="cuda", dtype=torch.float16)
    out = torch.full((T, Cc), float("nan"), device="cuda", dtype=torch.float16)
    cfg = (C.c_int32 * (4 * len(FIELDS)))()
    ctx.enter()
    ctx.check(lib.sdxl_dbg_plan_vae_attention(ctx.h, ptr(q), ptr(k), ptr(v), T, Cc, ptr(S), ptr(Pm), ptr(vT), ptr(out), cfg, 4),
              "sdxl_dbg_plan_vae_attention")
    ctx.leave()
    name = f"VAE attention T={T}"
    # S = q k^T in f32
    qd, kd, vd = q.double(), k.double(), v.double()
    check_bound(name + " scores", S, qd @ kd.T, qd.abs() @ kd.abs().T, Cc / 8 + 4)
    # softmax_rows on the kernel's own scores: f32 math, one f16 rounding of each probability
    Sd = S.double() / math.sqrt(Cc)
    Pref = torch.softmax(Sd, dim=-1)
    e = (Pm.double() - Pref).abs()
    worst = float((e / ((H16 + 2 ** -16) * Pref + 2 ** -24)).max())
    print(f"  {name} softmax_rows: worst |err|/bound {worst:.3f}")
    assert worst <= 1.0
    del Sd, Pref, e
    assert torch.equal(vT, v.T)
    # P v on the kernel's own probabilities, and the whole core against f64 attention
    ref = Pm.double() @ vd
    check_bound(name + " P v", out, ref, Pm.double().abs() @ vd.abs(), T / 8 + 4, f16_out=True)
    full = torch.softmax(qd @ kd.T / math.sqrt(Cc), dim=-1) @ vd
    check_attn(name, out[None], full[None], Cc // 64, ATTN_ROW_TOL["vae"])
    print("  PLANCFG " + json.dumps({"case": name, "cfg": [dict(zip(FIELDS, cfg[i * 8:(i + 1) * 8])) for i in range(2)]}))


# ---------------------------------------------------------------------------------------------------------------------------
AB_SETTINGS = {
    "pair0": ({"SDXL_B200_PAIR": "0"}, lambda c: c["pair"] == 0, None),
    "cluster2x2": ({"SDXL_B200_PAIR": "0", "SDXL_B200_CLUSTER": "2x2"}, lambda c: c["pair"] == 0,
                   lambda c: (c["CM"], c["CN"]) == (2, 2)),
    "epi_stg": ({"SDXL_B200_EPI_TMA": "0"}, lambda c: c["epi_tma"] == 0, None),
    "box_f32": ({"SDXL_B200_EPI_COMPACT": "0"}, lambda c: c["box"] == 4096, lambda c: c["epi_tma"] == 1),
}


@pytest.mark.parametrize("setting", list(AB_SETTINGS))
def test_ab_switch(setting):
    """The A/B switches of the GEMM launch structure, read once per process: the conv / linear sweep in a subprocess each, same
    bounds, and the forced variant must be what ran."""
    if FORCED:
        pytest.skip("already inside a forced-variant run")
    env_add, every, some = AB_SETTINGS[setting]
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, SDXL_B200_PLAN_TEST_FORCED=setting, **env_add)
    cmd = [sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", "-m", "gpu", os.path.abspath(__file__),
           "-k", "test_conv3 or test_upconv or test_head_hilo or test_padded_conv_s2 or test_linear"]
    r = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-2000:])
    cfgs = [c for ln in r.stdout.splitlines() if "PLANCFG " in ln for c in json.loads(ln.split("PLANCFG ", 1)[1])["cfg"]]
    print(f"  {setting}: {len(cfgs)} GEMM launches")
    assert len(cfgs) >= 30
    assert all(every(c) for c in cfgs), f"{setting}: a launch did not run the forced variant"
    if some:
        assert any(some(c) for c in cfgs)
