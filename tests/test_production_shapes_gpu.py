"""GPU tests at the shapes and batch sizes the engine runs in production (B = 32 utterances of 10 s per GPU and more).

Below that scale whole code paths of the kernels never run: a persistent conv-GEMM CTA never gets a second tile (tile
loop, TMEM accumulator ring, stage phases carried across tiles, the TMA epilogue's residual prefetch into the next tile),
and the GRU never groups more than 2 sequences per cluster.  Every case here mirrors a descriptor engine.cu issues.

Conv-GEMM cases run the tensor-core kernel (impl=1: a shape that left the tensor-core path fails as UNSUPPORTED) on
operands rounded to the storage format, against a float64 torch convolution of the same rounded values:
  * fp32 output, per element: |got - ref| <= 2 (K + 2) 2^-24 absref, absref = conv(|a|, |w|) + |bias| + |residual|,
    K = taps * Cin -- the worst case of fp32 accumulation in any order (the products of bf16 / fp16 / tf32 operands are
    exact in fp32), so one wrong element among millions fails; plus 2e-5 relative RMS over the tensor;
  * activated operand output, per element: one unit in the last place of the output format at |act|, plus
    Lip * |scale| * (the fp32 bound), plus 2e-6 (1 + |act|) for the fast intrinsics of the epilogue;
  * NaN sentinels wherever the kernel must not write (the other half of a concat buffer, pad rows, a batch row past B).
Cases marked multi-tile assert that every CTA runs more tiles than the TMEM accumulator ring holds, with a partial
last wave.  Run with -s to see the tile counts and the worst error / bound ratio of each case."""
import ctypes
import math
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from conftest import rel_rms

from voicefixer_b200 import _lib
from voicefixer_b200.weights import round_tf32

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U24 = 2.0 ** -24
PRECS = ["bf16", "tf32", "fp16"]
STORE = {"bf16": torch.bfloat16, "fp16": torch.float16, "tf32": torch.float32}
MANT = {"bf16": 7, "fp16": 10, "tf32": 10}            # explicit mantissa bits of the operand format
EMIN = {"bf16": -126, "fp16": -14, "tf32": -126}      # smallest normal exponent (below it the spacing is fixed)
LIP = {"lrelu": 1.0, "elu": 1.0, "lrelu_xsinx": 2.0, "sigmoid": 0.25}
TAPS3x3 = [(kh - 1, kw - 1) for kh in range(3) for kw in range(3)]


# ------------------------------------------------------------------------------------------------ operands and launch
def _gen(*shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


def _store(t, prec):
    """CPU fp32 tensor -> (the tensor in the storage format of `prec` on the GPU, its exact value in float64)."""
    q = (round_tf32(t) if prec == "tf32" else t.to(STORE[prec])).to(DEV)
    return q, q.double()


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


def _f32(x):
    return float(np.float32(x))


def _conv(prec, a, w, taps, N, w_off=None, Hq=None, Wq=None, sh=1, rh=0, sw=1, rw=0, OH=None, OW=None, bias=None,
          bias_mod=None, residual=None, out_raw=None, out_act=None, act="none", act_param=0.0, act_scale=None,
          act_shift=None, res_enc=0, raw_enc=0, enc_slope=0.0):
    """One vfx_conv_gemm call on the tensor-core kernel.  a, residual, out_raw, out_act: (B, H, W, C) views with unit
    channel stride, or (view, column offset) pairs; their pointers and strides go into the descriptor as they are."""
    lib = _lib.load()
    d = _lib.ConvDesc()
    B, H, W, Cin = a.shape
    d.a, d.B, d.H, d.W, d.Cin = a.data_ptr(), B, H, W, Cin
    d.a_sB, d.a_sH, d.a_sW = a.stride(0), a.stride(1), a.stride(2)
    d.w, d.ntaps = w.data_ptr(), len(taps)
    for i, (dh, dw) in enumerate(taps):
        d.dh[i], d.dw[i] = dh, dw
        d.w_off[i] = w_off[i] if w_off is not None else i * N * Cin
    d.Hq, d.Wq, d.N = Hq or H, Wq or W, N
    d.sh, d.rh, d.sw, d.rw = sh, rh, sw, rw
    d.OH, d.OW = OH or d.Hq, OW or d.Wq

    def view(t):
        t, col = t if isinstance(t, tuple) else (t, 0)
        assert t.stride(3) == 1
        return t.data_ptr(), t.stride(0), t.stride(1), t.stride(2), col
    if out_raw is not None:
        d.out_raw, d.o_sB, d.o_sH, d.o_sW, d.o_col = view(out_raw)
    if out_act is not None:
        d.out_act, d.oa_sB, d.oa_sH, d.oa_sW, d.oa_col = view(out_act)
    if residual is not None:
        d.residual, d.r_sB, d.r_sH, d.r_sW, d.r_col = view(residual)
    if bias is not None:
        d.bias, d.bias_mod = bias.data_ptr(), bias_mod or bias.numel()
    if act_scale is not None:
        d.act_scale, d.act_shift = act_scale.data_ptr(), act_shift.data_ptr()
    d.act, d.act_param = _lib.ACT[act], act_param
    d.res_enc, d.raw_enc, d.enc_slope = res_enc, raw_enc, enc_slope
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.vfx_conv_gemm(_lib.PREC[prec], 1, ctypes.byref(d), st), "vfx_conv_gemm")
    torch.cuda.synchronize()


def _w3x3(w):
    """(Cout, Cin, 3, 3) -> the kernel's [tap][Cout][Cin]."""
    return w.permute(2, 3, 0, 1).reshape(9, w.shape[0], w.shape[1]).contiguous()


# ------------------------------------------------------------------------------------------------ tile schedule
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _regime(tag, B, Hq, Wq, N, multi):
    """The host tiling of conv_gemm_tc.cu: 128-position tiles of tw x th, N tiles of the widest of 256/128/64/32 dividing N,
    512 / Ntile TMEM accumulator stages (at most 8), one persistent CTA per SM.  A multi-tile case must give every CTA more
    tiles than the accumulator ring holds, and leave a partial last wave."""
    tw = 1
    while tw < Wq and tw < 128:
        tw *= 2
    th = 128 // tw
    ntile = next(c for c in (256, 128, 64, 32) if N % c == 0)
    nacc = min(8, 512 // ntile)
    tiles = B * -(-Hq // th) * -(-Wq // tw) * (N // ntile)
    sms = _sms()
    if multi:
        assert tiles >= sms * (nacc + 1) + 1 and tiles % sms != 0, \
            f"{tag}: {tiles} tiles on {sms} SMs (nacc {nacc}) is not the multi-tile regime"
    return f"tiles {tiles} ({tiles / sms:.1f} per CTA, nacc {nacc})"


# ------------------------------------------------------------------------------------------------ bounds
def _ulp(x, prec):
    e = torch.floor(torch.log2(x.abs().clamp_min(1e-300))).clamp_min(EMIN[prec])
    return torch.exp2(e - MANT[prec])


def _act64(v, act, p):
    if act == "lrelu":
        return torch.where(v > 0, v, v * p)
    if act == "elu":
        return torch.where(v > 0, v, torch.expm1(v))
    if act == "lrelu_xsinx":
        u = torch.where(v > 0, v, v * p)
        return u + torch.sin(u)
    assert act == "sigmoid"
    return torch.sigmoid(v)


def _worst(tag, what, got, ref, bound):
    """max |got - ref| / bound; fails on the first element outside the bound (NaN included)."""
    err = (got.double() - ref).abs()
    ok = err <= bound
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{tag}: {what}: {bad.shape[0]} of {ok.numel()} elements outside the bound, first at {i}: "
                             f"got {float(got[i]):.9g} ref {float(ref[i]):.9g} bound {float(bound[i]):.3g}")
    return float((err / bound).max())


def _check_raw(tag, got, ref, absref, K, extra=0.0):
    """fp32 output: worst-case accumulation bound per element, 2e-5 relative RMS overall.  Returns (worst ratio, bound)."""
    rb = 2 * (K + 2) * U24 * absref + 1e-30
    worst = _worst(tag, "fp32 output", got, ref, rb + extra)
    d = got.double() - ref
    assert float(d.square().mean().sqrt() / ref.square().mean().sqrt()) < 2e-5, tag
    return worst, rb


def _check_act(tag, prec, got, act64, act, scale_abs, rb):
    bound = _ulp(act64, prec) + LIP[act] * scale_abs * rb + 2e-6 * (1 + act64.abs())
    worst = _worst(tag, "activated output", got, act64, bound)
    if prec == "tf32":      # the operand output is exactly representable in tf32 (low 13 mantissa bits zero)
        assert int((got.view(torch.int32) & 0x1FFF).abs().max()) == 0, tag
    return worst


def _still_nan(tag, t, what):
    n = int((~torch.isnan(t.float())).sum())
    assert n == 0, f"{tag}: {n} elements written into {what}"


def _report(tag, regime, **worst):
    print(f"\n[{tag}] {regime}; worst err/bound " + " ".join(f"{k} {v:.3f}" for k, v in worst.items()), end="")


def _conv2d64(a64, w64, **kw):
    """float64 conv2d of channels-last a (B, H, W, C), channels-last result; and the same of |a|, |w|."""
    f = lambda x, y: F.conv2d(x.permute(0, 3, 1, 2), y, **kw).permute(0, 2, 3, 1)
    return f(a64, w64), f(a64.abs(), w64.abs())


def _conv1d64(a64, w64, **kw):
    """float64 conv1d of channels-last a (B, 1, L, C) -> (B, 1, L', N); and the same of |a|, |w|."""
    f = lambda x, y: F.conv1d(x[:, 0].permute(0, 2, 1), y, **kw).permute(0, 2, 1)[:, None]
    return f(a64, w64), f(a64.abs(), w64.abs())


def _bn_affine(C, seed):
    """A folded eval-mode BatchNorm: per-channel scale and shift."""
    return torch.exp(_gen(C, seed=seed, scale=0.3)).to(DEV), _gen(C, seed=seed + 1, scale=0.5).to(DEV)


# ================================================================================================ A. conv-GEMM
# UNet conv2 of a ConvBlockRes (engine.cu conv_block): 3x3 C -> C, residual = the block input, fp32 result written over it
# in place, and the NEXT block's operand act(bn1(result)) from the same epilogue (eval BatchNorm fused as act_scale /
# act_shift; slope 0.01 = LeakyReLU, 0 = the ReLU before a decoder's ConvTranspose).  Encoder levels live in the second
# half of the decoder's concat buffer (pitch 2C); the centre block works at W = 1 on a dense tensor.
# (name, B, H, W, C, slope, in the concat buffer, multi-tile)
UNET_CONV2 = [("enc1", 2, 1024, 127, 32, 0.01, True, True), ("enc2", 6, 512, 63, 64, 0.01, True, True),
              ("enc3", 12, 256, 31, 128, 0.01, True, True), ("enc3_relu", 12, 256, 31, 128, 0.0, True, True),
              ("enc4", 29, 128, 15, 256, 0.01, True, True), ("enc5", 62, 64, 7, 384, 0.01, True, True),
              ("enc6", 248, 32, 3, 384, 0.01, True, True), ("centre", 32, 16, 1, 384, 0.0, False, False)]


@pytest.mark.parametrize("name,B,H,W,C,slope,concat,multi", UNET_CONV2, ids=[c[0] for c in UNET_CONV2])
@pytest.mark.parametrize("prec", PRECS)
def test_unet_conv2_residual_in_place(name, B, H, W, C, slope, concat, multi, prec):
    tag = f"unet conv2 {name} {prec}"
    regime = _regime(tag, B, H, W, C, multi)
    s = sum(map(ord, name))
    a, a64 = _store(_gen(B, H, W, C, seed=s), prec)
    w, w64 = _store(_gen(C, C, 3, 3, seed=s + 1, scale=1.5 / math.sqrt(9 * C)), prec)
    res = _gen(B, H, W, C, seed=s + 2).to(DEV)
    scale, shift = _bn_affine(C, s + 3)
    buf = _nan(B + 1, H, W, 2 * C if concat else C)
    x = buf[:B, ..., C:] if concat else buf[:B]
    x.copy_(res)
    op = _nan(B + 1, H, W, C, dtype=STORE[prec])
    _conv(prec, a, _w3x3(w), TAPS3x3, C, residual=x, out_raw=x, out_act=op[:B], act="lrelu", act_param=slope,
          act_scale=scale, act_shift=shift)
    conv, aconv = _conv2d64(a64, w64, padding=1)
    ref = conv + res.double()
    wr, rb = _check_raw(tag, x, ref, aconv + res.double().abs(), 9 * C)
    act = _act64(ref * scale.double() + shift.double(), "lrelu", _f32(slope))
    wa = _check_act(tag, prec, op[:B], act, "lrelu", scale.double().abs(), rb)
    if concat:
        _still_nan(tag, buf[..., :C], "the first half of the concat buffer")
    _still_nan(tag, buf[B], "the batch row past B")
    _still_nan(tag, op[B], "the operand's batch row past B")
    _report(tag, regime, raw=wr, act=wa)


# First encoder block (2 input channels zero-padded to 32 operand channels) and the first block of a decoder level (2C -> C
# from the concat buffer): conv1 (3x3 + bias, LeakyReLU operand out), the 1x1 shortcut (bias, fp32 out), then conv2 on
# conv1's output with the shortcut as residual, into the skip half of a concat buffer (first block) or a dense tensor.
@pytest.mark.parametrize("block", ["first", "decoder"])
@pytest.mark.parametrize("prec", PRECS)
def test_unet_block_conv1_shortcut_conv2(block, prec):
    if block == "first":
        B, H, W, Cin, Cop, C, concat = 2, 1024, 127, 2, 32, 32, True
    else:
        B, H, W, Cin, Cop, C, concat = 6, 512, 63, 128, 128, 64, False
    tag = f"unet {block} block {prec}"
    regime = _regime(tag, B, H, W, C, True)
    s = 500 if block == "first" else 600
    pad = lambda t: torch.cat([t[..., :Cin], torch.zeros_like(t[..., Cin:])], -1) if Cin < Cop else t

    def padw(t):
        t = t.clone()
        t[:, Cin:] = 0
        return t
    a1, a1_64 = _store(pad(_gen(B, H, W, Cop, seed=s)), prec)
    ax, ax64 = _store(pad(_gen(B, H, W, Cop, seed=s + 1)), prec)
    w1, w1_64 = _store(padw(_gen(C, Cop, 3, 3, seed=s + 2, scale=1.5 / math.sqrt(9 * Cin))), prec)
    wsc, wsc64 = _store(padw(_gen(C, Cop, 1, 1, seed=s + 3, scale=1.0 / math.sqrt(Cin))), prec)
    w2, w2_64 = _store(_gen(C, C, 3, 3, seed=s + 4, scale=1.5 / math.sqrt(9 * C)), prec)
    b1, bsc = _gen(C, seed=s + 5).to(DEV), _gen(C, seed=s + 6).to(DEV)
    scale, shift = _bn_affine(C, s + 7)
    # conv1: h = lrelu(conv1(a) + b1), operand out only
    h = _nan(B + 1, H, W, C, dtype=STORE[prec])
    _conv(prec, a1, _w3x3(w1), TAPS3x3, C, bias=b1, out_act=h[:B], act="lrelu", act_param=0.01)
    conv, aconv = _conv2d64(a1_64, w1_64, padding=1)
    rb = 2 * (9 * Cop + 2) * U24 * (aconv + b1.double().abs()) + 1e-30
    w_h = _check_act(tag + " conv1", prec, h[:B], _act64(conv + b1.double(), "lrelu", _f32(0.01)), "lrelu", 1.0, rb)
    _still_nan(tag, h[B], "conv1's batch row past B")
    # shortcut: 1x1 + bias, fp32 out
    rs = _nan(B + 1, H, W, C)
    _conv(prec, ax, wsc[:, :, 0, 0].contiguous(), [(0, 0)], C, bias=bsc, out_raw=rs[:B])
    conv, aconv = _conv2d64(ax64, wsc64)
    w_s, _ = _check_raw(tag + " shortcut", rs[:B], conv + bsc.double(), aconv + bsc.double().abs(), Cop)
    _still_nan(tag, rs[B], "the shortcut's batch row past B")
    # conv2 on conv1's output, shortcut as residual, fused next BatchNorm + LeakyReLU operand
    buf = _nan(B + 1, H, W, 2 * C if concat else C)
    out = buf[:B, ..., C:] if concat else buf[:B]
    op = _nan(B + 1, H, W, C, dtype=STORE[prec])
    _conv(prec, h[:B], _w3x3(w2), TAPS3x3, C, residual=rs[:B], out_raw=out, out_act=op[:B], act="lrelu",
          act_param=0.01, act_scale=scale, act_shift=shift)
    conv, aconv = _conv2d64(h[:B].double(), w2_64, padding=1)
    r64 = rs[:B].double()
    ref = conv + r64
    w_r, rb = _check_raw(tag + " conv2", out, ref, aconv + r64.abs(), 9 * C)
    act = _act64(ref * scale.double() + shift.double(), "lrelu", _f32(0.01))
    w_a = _check_act(tag + " conv2", prec, op[:B], act, "lrelu", scale.double().abs(), rb)
    if concat:
        _still_nan(tag, buf[..., :C], "the first half of the concat buffer")
    _still_nan(tag, buf[B], "the batch row past B")
    _still_nan(tag, op[B], "the operand's batch row past B")
    _report(tag, regime, conv1_act=w_h, shortcut=w_s, conv2_raw=w_r, conv2_act=w_a)


# ConvTranspose2d(k3, s2) of a decoder level as four output-parity GEMMs (direct epilogue) into the first half of the
# concat buffer, at the decoder's production grids: input W 1, 3, 7, 15, 31, 63 -> output 2W + 1, height 2H (last row pruned).
# (Cin, Cout, H, W, B)
CONVT = [(384, 384, 16, 1, 32), (384, 384, 32, 3, 16), (384, 256, 64, 7, 8), (256, 128, 128, 15, 4),
         (128, 64, 256, 31, 2), (64, 32, 512, 63, 2)]


@pytest.mark.parametrize("Cin,Cout,H,W,B", CONVT)
@pytest.mark.parametrize("prec", PRECS)
def test_unet_conv_transpose_into_concat_buffer(Cin, Cout, H, W, B, prec):
    tag = f"unet convT {Cin}->{Cout} W{W}->{2 * W + 1} {prec}"
    regime = _regime(tag, B, H, W + 1, Cout, False)
    x, x64 = _store(_gen(B, H, W, Cin, seed=700 + W), prec)
    w, w64 = _store(_gen(Cin, Cout, 3, 3, seed=701 + W, scale=1.5 / math.sqrt(4 * Cin)), prec)
    OH, OW = 2 * H, 2 * W + 1
    wk = w.permute(2, 3, 1, 0).reshape(9, Cout, Cin).contiguous()
    cat = _nan(B + 1, OH, OW, 2 * Cout)
    for rh in range(2):
        for rw in range(2):
            taps, offs = [], []
            for kh in ([1] if rh else [0, 2]):
                for kw in ([1] if rw else [0, 2]):
                    taps.append((-1 if kh == 2 else 0, -1 if kw == 2 else 0))
                    offs.append((kh * 3 + kw) * Cout * Cin)
            _conv(prec, x, wk, taps, Cout, w_off=offs, Hq=H, Wq=W + 1, sh=2, rh=rh, sw=2, rw=rw, OH=OH, OW=OW,
                  out_raw=cat[:B, ..., :Cout])
    f = lambda a, b: F.conv_transpose2d(a.permute(0, 3, 1, 2), b, stride=2)[:, :, :-1, :].permute(0, 2, 3, 1)
    wr, _ = _check_raw(tag, cat[:B, ..., :Cout], f(x64, w64), f(x64.abs(), w64.abs()), 4 * Cin)
    _still_nan(tag, cat[..., Cout:], "the second half of the concat buffer")
    _still_nan(tag, cat[B], "the batch row past B")
    _report(tag, regime, raw=wr)


# Denoiser linears (engine.cu linear / bn_gru): one GEMM over M = B * T rows (H = 1, W = M), bias, fp32 out.  At B = 32,
# T = 1001 the 512- and 1536-wide ones are multi-tile; 1536 = 6 N tiles (weights streamed, not resident).
LINEARS = [(128, 256), (256, 512), (512, 1536), (512, 512), (512, 128)]


@pytest.mark.parametrize("M", [32 * 1001, 63, 1])
@pytest.mark.parametrize("K,N", LINEARS)
@pytest.mark.parametrize("prec", PRECS)
def test_denoiser_linear(K, N, M, prec):
    tag = f"linear {K}->{N} M={M} {prec}"
    regime = _regime(tag, 1, 1, M, N, M > 10000 and N >= 512)
    a, a64 = _store(_gen(1, 1, M, K, seed=800 + K), prec)
    w, w64 = _store(_gen(N, K, seed=801 + N, scale=1.0 / math.sqrt(K)), prec)
    b = _gen(N, seed=802).to(DEV)
    out = _nan(2, 1, M + 1, N)                  # a batch row and a position row past the output as sentinels
    _conv(prec, a, w, [(0, 0)], N, bias=b, out_raw=out[:1, :, :M])
    ref, aref = a64 @ w64.t() + b.double(), a64.abs() @ w64.abs().t() + b.double().abs()
    wr, _ = _check_raw(tag, out[:1, :, :M], ref, aref, K)
    _still_nan(tag, out[:1, :, M], "the row past M")
    _still_nan(tag, out[1], "the batch row past B")
    _report(tag, regime, raw=wr)


# Vocoder condnet (engine.cu:514-532): Conv1d(k3, p1) + bias + ELU, operand out only, B = 32, Tc = 1006.  The last layer
# writes rows 3 .. Tc+2 of the (Tc + 6)-row reflect-pad buffer (item stride (Tc + 6) * 512); the pad rows are sentinels.
@pytest.mark.parametrize("Cin,last", [(128, False), (512, True)])
@pytest.mark.parametrize("prec", PRECS)
def test_condnet_elu_into_padded_buffer(Cin, last, prec):
    B, Tc, N = 32, 1006, 512
    tag = f"condnet {Cin}->{N} {'padded' if last else 'dense'} {prec}"
    regime = _regime(tag, B, 1, Tc, N, True)
    a, a64 = _store(_gen(B, 1, Tc, Cin, seed=900 + Cin), prec)
    w, w64 = _store(_gen(N, Cin, 3, seed=901 + Cin, scale=2.0 / math.sqrt(3 * Cin)), prec)
    b = _gen(N, seed=902).to(DEV)
    rows = Tc + 6 if last else Tc
    buf = _nan(B + 1, 1, rows, N, dtype=STORE[prec])
    out = buf[:B, :, 3:Tc + 3] if last else buf[:B]
    _conv(prec, a, w.permute(2, 0, 1).contiguous(), [(0, -1), (0, 0), (0, 1)], N, bias=b, out_act=out, act="elu")
    conv, aconv = _conv1d64(a64, w64, padding=1)
    rb = 2 * (3 * Cin + 2) * U24 * (aconv + b.double().abs()) + 1e-30
    wa = _check_act(tag, prec, out, _act64(conv + b.double(), "elu", 0.0), "elu", 1.0, rb)
    if last:
        _still_nan(tag, buf[:B, :, :3], "the leading pad rows")
        _still_nan(tag, buf[:B, :, Tc + 3:], "the trailing pad rows")
    _still_nan(tag, buf[B], "the batch row past B")
    _report(tag, regime, act=wa)


# Vocoder pre-conv (engine.cu:536-543): k7 'valid' 512 -> 1024 on the padded condnet output, LeakyReLU(0.2) followed by
# x + sin x in the epilogue.  Pre-activations reach |u| ~ 60, so the Cody-Waite reduction of the sine runs with k != 0.
@pytest.mark.parametrize("prec", PRECS)
def test_vocoder_preconv_xsinx(prec):
    B, Tc, Cin, N = 32, 1006, 512, 1024
    tag = f"voc pre-conv {prec}"
    regime = _regime(tag, B, 1, Tc, N, True)
    a, a64 = _store(_gen(B, 1, Tc + 6, Cin, seed=1000), prec)
    w, w64 = _store(_gen(N, Cin, 7, seed=1001, scale=10.0 / math.sqrt(7 * Cin)), prec)
    b = _gen(N, seed=1002, scale=2.0).to(DEV)
    buf = _nan(B + 1, 1, Tc, N, dtype=STORE[prec])
    _conv(prec, a, w.permute(2, 0, 1).contiguous(), [(0, k) for k in range(7)], N, Wq=Tc, OW=Tc, bias=b, out_act=buf[:B],
          act="lrelu_xsinx", act_param=0.2)
    conv, aconv = _conv1d64(a64, w64)
    v = conv + b.double()
    u_max = float(torch.where(v > 0, v, v * 0.2).abs().max())
    assert 32 < u_max <= 80, u_max
    rb = 2 * (7 * Cin + 2) * U24 * (aconv + b.double().abs()) + 1e-30
    wa = _check_act(tag, prec, buf[:B], _act64(v, "lrelu_xsinx", _f32(0.2)), "lrelu_xsinx", 1.0, rb)
    _still_nan(tag, buf[B], "the batch row past B")
    _report(tag, regime + f", max |u| {u_max:.1f}", act=wa)


# UpsampleNet ConvTranspose1d(k = 2u, s = u) as two phase-group GEMMs (engine.cu:555-580): the output is the reshaped view
# [B][Lin][u * Co]; group 0 writes columns [0, nA Co), group 1 [nA Co, u Co), fp32 result plus the LeakyReLU operand, both
# at column offset r0 * Co of a u * Co pitch.  (Cin, Cout, u) of VOC_CIN / VOC_COUT / VOC_U, B, Lin
UPSAMPLERS = [(1024, 512, 7, 8, 1006), (512, 256, 7, 4, 2000), (256, 128, 3, 4, 4000), (128, 64, 3, 4, 8000)]


@pytest.mark.parametrize("Ci,Co,u,B,Lin", UPSAMPLERS)
@pytest.mark.parametrize("prec", PRECS)
def test_upsampler_phase_groups_pitched(Ci, Co, u, B, Lin, prec):
    tag = f"voc up {Ci}->{Co} u{u} {prec}"
    x, x64 = _store(_gen(B, 1, Lin, Ci, seed=1100 + Ci), prec)
    w, w64 = _store(_gen(Ci, Co, 2 * u, seed=1101 + Ci, scale=1.5 / math.sqrt(2 * Ci)), prec)
    b = _gen(Co, seed=1102).to(DEV)
    pad, mat = u // 2 + u % 2, Co * Ci
    nA = u - pad
    wk = w.permute(2, 1, 0).contiguous()                 # (2u, Co, Ci)
    X = _nan(B + 1, 1, Lin, u * Co)
    A = _nan(B + 1, 1, Lin, u * Co, dtype=STORE[prec])
    regimes = []
    for grp in range(2):
        nph = nA if grp == 0 else u - nA
        r0 = 0 if grp == 0 else nA
        regimes.append(_regime(tag, B, 1, Lin, nph * Co, False))
        taps, offs = ([(0, 0), (0, -1)], [pad * mat, (pad + u) * mat]) if grp == 0 else ([(0, 1), (0, 0)], [0, u * mat])
        _conv(prec, x, wk, taps, nph * Co, w_off=offs, bias=b, bias_mod=Co, out_raw=(X[:B], r0 * Co),
              out_act=(A[:B], r0 * Co), act="lrelu", act_param=0.01)
        if grp == 0:
            _still_nan(tag, X[:B, ..., nA * Co:], "phase group 1's columns (raw) after group 0")
            _still_nan(tag, A[:B, ..., nA * Co:], "phase group 1's columns (operand) after group 0")
    f = lambda a, c: F.conv_transpose1d(a[:, 0].permute(0, 2, 1), c, stride=u, padding=pad, output_padding=u % 2)
    to_view = lambda y: y.permute(0, 2, 1).reshape(B, 1, Lin, u * Co)
    ref = to_view(f(x64, w64) + b.double()[:, None])
    aref = to_view(f(x64.abs(), w64.abs()) + b.double().abs()[:, None])
    wr, rb = _check_raw(tag, X[:B], ref, aref, 2 * Ci)
    wa = _check_act(tag, prec, A[:B], _act64(ref, "lrelu", _f32(0.01)), "lrelu", 1.0, rb)
    _still_nan(tag, X[B], "the batch row past B")
    _still_nan(tag, A[B], "the operand's batch row past B")
    _report(tag, " / ".join(regimes), raw=wr, act=wa)


@pytest.mark.parametrize("prec", PRECS)
def test_sigmoid_epilogue(prec):
    """VFX_ACT_SIGMOID is in the ABI and compiled for every format: k3 conv 64 -> 128, bias, fp32 and operand out."""
    B, L, Cin, N = 2, 3000, 64, 128
    tag = f"sigmoid {prec}"
    regime = _regime(tag, B, 1, L, N, False)
    a, a64 = _store(_gen(B, 1, L, Cin, seed=1200), prec)
    w, w64 = _store(_gen(N, Cin, 3, seed=1201, scale=3.0 / math.sqrt(3 * Cin)), prec)
    b = _gen(N, seed=1202).to(DEV)
    raw, op = _nan(B + 1, 1, L, N), _nan(B + 1, 1, L, N, dtype=STORE[prec])
    _conv(prec, a, w.permute(2, 0, 1).contiguous(), [(0, -1), (0, 0), (0, 1)], N, bias=b, out_raw=raw[:B],
          out_act=op[:B], act="sigmoid")
    conv, aconv = _conv1d64(a64, w64, padding=1)
    ref = conv + b.double()
    wr, rb = _check_raw(tag, raw[:B], ref, aconv + b.double().abs(), 3 * Cin)
    wa = _check_act(tag, prec, op[:B], _act64(ref, "sigmoid", 0.0), "sigmoid", 1.0, rb)
    _still_nan(tag, raw[B], "the batch row past B")
    _still_nan(tag, op[B], "the operand's batch row past B")
    _report(tag, regime, raw=wr, act=wa)


# ResStack conv2 residual forms at width 64 (the epilogue warp layouts: 16-bit operands with a residual use 4 warps and a
# 4-slot residual ring, tf32 uses 8 warps and 2 slots).  plain: fp32 residual stream x, x' = x + conv(h) + b written over
# it in place, lrelu(x') operand out.  enc (tf32): x travels as the encoded stream S = bits(lrelu(x, 0.01)) + 0x1000,
# decoded as the residual and re-encoded in place (res_enc / raw_enc).
RES_FORMS = [(f, p, d) for f, ps in (("plain", PRECS), ("enc", ["tf32"])) for p in ps for d in (1, 81, 2187)]


def _enc(x):
    y = torch.where(x > 0, x, x * _f32(0.01))
    return (y.view(torch.int32) + 0x1000).view(torch.float32)


@pytest.mark.parametrize("form,prec,dil", RES_FORMS)
def test_resstack_residual_forms(form, prec, dil):
    B, L, C = 4, 48000, 64
    tag = f"resstack conv2 {form} d{dil} {prec}"
    regime = _regime(tag, B, 1, L, C, True)
    h, h64 = _store(_gen(B, 1, L, C, seed=1300 + dil), prec)
    w, w64 = _store(_gen(C, C, 3, seed=1301 + dil, scale=1.5 / math.sqrt(3 * C)), prec)
    b = _gen(C, seed=1302).to(DEV)
    x = _gen(B, 1, L, C, seed=1303 + dil).to(DEV)
    taps = [(0, -dil), (0, 0), (0, dil)]
    wk = w.permute(2, 0, 1).contiguous()
    buf = _nan(B + 1, 1, L, C)
    conv, aconv = _conv1d64(h64, w64, padding=dil, dilation=dil)
    if form == "plain":
        buf[:B] = x
        op = _nan(B + 1, 1, L, C, dtype=STORE[prec])
        _conv(prec, h, wk, taps, C, bias=b, residual=buf[:B], out_raw=buf[:B], out_act=op[:B], act="lrelu",
              act_param=0.01)
        ref = conv + b.double() + x.double()
        wr, rb = _check_raw(tag, buf[:B], ref, aconv + b.double().abs() + x.double().abs(), 3 * C)
        wa = _check_act(tag, prec, op[:B], _act64(ref, "lrelu", _f32(0.01)), "lrelu", 1.0, rb)
        _still_nan(tag, op[B], "the operand's batch row past B")
        worst = dict(raw=wr, act=wa)
    else:
        buf[:B] = _enc(x)
        y = (buf[:B].view(torch.int32) - 0x1000).view(torch.float32)
        xr = torch.minimum(y, y * _f32(100.0)).double()          # the residual exactly as the kernel decodes it
        _conv(prec, h, wk, taps, C, bias=b, residual=buf[:B], out_raw=buf[:B], res_enc=1, raw_enc=1, enc_slope=0.01)
        yo = (buf[:B].view(torch.int32) - 0x1000).view(torch.float32).double()
        got = torch.where(yo > 0, yo, yo / _f32(0.01))            # exact inverse of the encoder's slope multiply
        ref = conv + b.double() + xr
        absref = aconv + b.double().abs() + xr.abs()
        wr, _ = _check_raw(tag, got, ref, absref, 3 * C, extra=U24 * absref)   # + the encoder's one rounding
        worst = dict(raw=wr)
    _still_nan(tag, buf[B], "the batch row past B")
    _report(tag, regime, **worst)


# ================================================================================================ B. GRU recurrence
# gru.cu groups G sequences per 8-CTA cluster: B <= 16 -> G = 2, B <= 32 -> G = 4, else G = 8.  (B, T) covers every G,
# partial last groups and the edges of the two-step gi prefetch ring.  Error against a float64 torch.nn.GRU on the same
# (fp32-valued) weights, measured on one B200 (1000 W): relative RMS 7.2e-8 .. 8.7e-8, max |err| 7.6e-8 .. 2.2e-7 over all
# eight cases -- it does not grow with T (1001 steps: 8.7e-8 / 2.2e-7).  The bounds keep a margin of more than 4x.
GRU_CASES = [(1, 1), (2, 2), (16, 3), (17, 37), (32, 1001), (33, 37), (64, 1001), (64, 1)]
GRU_TOL_RMS, GRU_TOL_MAX = 4e-7, 1e-6


@pytest.mark.parametrize("B,T", GRU_CASES)
def test_gru_layer_every_grouping(B, T):
    lib = _lib.load()
    torch.manual_seed(7)
    gru = torch.nn.GRU(512, 256, num_layers=1, bidirectional=True, batch_first=True).double()   # fp32-valued weights
    x = _gen(B, T, 512, seed=1400 + B + T).double()
    with torch.no_grad():
        ref, _ = gru(x)
        wih = torch.cat([gru.weight_ih_l0, gru.weight_ih_l0_reverse], 0).to(DEV)
        bih = torch.cat([gru.bias_ih_l0, gru.bias_ih_l0_reverse], 0).to(DEV)
        gi = (x.to(DEV) @ wih.t() + bih).float().contiguous()                      # [B][T][2][768]
        whh_t = torch.stack([gru.weight_hh_l0.t(), gru.weight_hh_l0_reverse.t()], 0).float().contiguous().to(DEV)
        bhh = torch.stack([gru.bias_hh_l0, gru.bias_hh_l0_reverse], 0).float().contiguous().to(DEV)
    out = _nan(B + 1, T, 512)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    _lib.check(lib.vfx_gru_layer(p(gi), p(whh_t), p(bhh), B, T, p(out), None), "vfx_gru_layer")
    torch.cuda.synchronize()
    got = out[:B].double().cpu()
    err_rms = rel_rms(got.numpy(), ref.numpy())
    err_max = float((got - ref).abs().max())
    G = 2 if B <= 16 else 4 if B <= 32 else 8
    print(f"\n[gru B={B} T={T} G={G}] rel-RMS {err_rms:.3e}, max |err| {err_max:.3e}", end="")
    assert err_rms < GRU_TOL_RMS and err_max < GRU_TOL_MAX, (err_rms, err_max)
    _still_nan(f"gru B={B}", out[B], "the sequence row past B")


# ================================================================================================ C. engine at production batch
# B = 32 (GRU groups of 4) and B = 33 (groups of 8, the last one partial) utterances of 10 s.  Items restored alone equal
# their batch rows; the seed-1234 utterance, placed last, matches the CPU oracle at the precision's full-size tolerance
# (test_parity_gpu.FULL_TOL); at B = 32 one replay of the captured CUDA graph equals a direct restore.


@pytest.fixture(scope="module")
def production_batch(states):
    from voicefixer_b200 import synthetic
    from oracle import vf_oracle as O
    wav = synthetic.make_utterances(1, seconds=10.0, seed=1234)[0]
    ref = O.restore_inmem(wav, states[0], states[1], mode=0)
    others = synthetic.make_utterances(32, seconds=10.0, seed=2026)
    return others, wav, ref


@pytest.fixture(scope="module")
def engine_cache():
    cache = {}
    yield cache
    cache.clear()
    torch.cuda.empty_cache()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("prec,B", [(p, b) for p in PRECS for b in (32, 33)])
def test_engine_production_batch(states, production_batch, engine_cache, prec, B):
    from voicefixer_b200.engine import Engine
    from test_parity_gpu import FULL_TOL
    others, wav, ref = production_batch
    if prec not in engine_cache:              # one engine (and workspace) alive at a time
        engine_cache.clear()
        torch.cuda.empty_cache()
        engine_cache[prec] = Engine(states[0], states[1], precision=prec)
    eng = engine_cache[prec]
    t0 = time.perf_counter()
    batch = torch.from_numpy(np.concatenate([others[:B - 1], wav[None]])).to(DEV)
    y = eng.restore(batch).clone()
    max_diff = 0.0
    for i in (0, 1, 16, B - 2, B - 1):
        yi = eng.restore(batch[i:i + 1])
        assert rel_rms(yi.cpu().numpy(), y[i:i + 1].cpu().numpy()) < 1e-6, (prec, B, i)
        max_diff = max(max_diff, float((yi[0] - y[i]).abs().max()))
    last = y[B - 1:].cpu().numpy()
    tol_rms, tol_mae = FULL_TOL[prec]
    err = rel_rms(last, ref)
    assert err < tol_rms and float(np.mean(np.abs(last - ref))) < tol_mae, (prec, B, err)
    graph = ""
    if B == 32:
        out = torch.empty_like(batch)
        g = eng.make_graph(batch, out)
        direct = eng.restore(batch).clone()
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, direct), prec
        graph = ", graph replay == direct"
        del g
    print(f"\n[engine {prec} B={B}] single items vs batch rows: max |diff| {max_diff:.3e}; last item vs oracle rel-RMS "
          f"{err:.3e}{graph} ({time.perf_counter() - t0:.1f} s)", end="")
