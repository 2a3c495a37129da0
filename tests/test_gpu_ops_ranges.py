"""GPU: the operators outside unit-variance inputs.  tests/test_gpu_ops.py checks shapes with randn data; here the VALUES go where the
kernels' accuracy depends on them -- peaked / shifted softmax rows, activations from 1e-5 to 3e4 through the fp16 / E4M3 operand splits,
strided tensor-core outputs, and the edge cases of the row ops (NaN / inf durations, out-of-range ids, numpy's int16 cast).

Every bar is the kernel's documented error model evaluated on the test's own data in fp64 (the arithmetic is in each docstring), not a
number fitted to the observed error.  fp32 unit roundoff u = 2^-24; one ulp of a running fp32 sum is at most 2^-23 of its magnitude."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from fastspeech2_b200 import _lib as L, ops, packing
from tests import emul_cabi as E

pytestmark = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24
SCALES = [1e-5, 1e-2, 1.0, 100.0, 300.0, 500.0, 3e4]
F16_MAX = 65504.0
F8_SAT = 256.0          # from |a| = 256 the E4M3 byte of a_lo * 2^12 can pass 448 (fp16 half-ulp there is 0.125)


def g(seed=0):
    return torch.Generator().manual_seed(seed)


def rnd(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=g(seed)) * scale


def lin(a, w, dil=1, pad=0):
    """The conv's tap / channel sums without bias or activations (fp64 when a and w are)."""
    return E.conv1d(a, w, None, dil, pad, 0, 0.0, 0, 0.0, None, 1.0, None, None)


# ------------------------------------------------------------------------------------------------ split-operand emulation
def _f16(t):
    """fp32 -> fp16 round-to-nearest, saturating at +-65504 (cvt.rn.satfinite.f16x2.f32), back to fp32."""
    return t.float().clamp(-F16_MAX, F16_MAX).half().float()


def _e4(t):
    """fp32 -> E4M3 round-to-nearest, saturating at +-448 (cvt.rn.satfinite.e4m3x2.f32), back to fp32."""
    return t.float().clamp(-448, 448).to(torch.float8_e4m3fn).float()


def _split_operands(x, w, in_act, in_slope, f8):
    """The operands the tcgen05 kernel multiplies, evaluated exactly (a copy of test_gpu_ops.py::_f8_operand_emulation, extended with
    the fp16 saturation of the activation split and with the three-MMA format): returns (a, [(a_part, w_part)], s) in fp64 so that
    y * s = sum a_part . w_part  (conv_tc_kernel.cuh::tc_convert_store, packing.pack_conv_tc)."""
    a = x.float()
    if in_act == 3:
        a = torch.maximum(a, a * in_slope)
    ah = _f16(a)
    al = a - ah                                             # exact in fp32, as in the kernel
    hi, lo, s = packing.split_fp16(w)
    if f8:
        wl = w.float() * s - hi.float()
        parts = [(ah, hi.float()), (_e4(al * 4096.0) / 4096.0, _e4(hi.float() * 2.0 ** -12) * 4096.0), (_e4(ah), _e4(wl))]
    else:
        parts = [(ah, hi.float()), (_f16(al), hi.float()), (ah, lo.float())]
    return a.double(), [(p.double(), q.double()) for p, q in parts], s


def tc_model(x, w, *, dil=1, pad=0, in_act=0, in_slope=0.0, f8=False, segments=False):
    """fp64 model of the tensor-core conv's pre-activation (no bias).  Returns (contract, acc_bound, op_bound, saturated):
      contract   the exactly rounded operand products the kernel multiplies, summed in fp64;
      acc_bound  what the truncating fp32 accumulator may add to it: <= 1 ulp (2^-23 relative) of the running sum per MMA, the running sum
                 bounded by sum |a_part||w_part|; 3 MMAs per K = 16 step for the three-MMA split, 2 for f16 + f8 (one K = 32 f8f6f4
                 MMA).  K-segmented: a fresh 16-step chain per (tap, 256-channel) segment plus one fp32 round-to-nearest add per segment;
      op_bound   |contract - exact|, per product a.w:
                   three-MMA: 4 * 2^-22 |a||w| (fp16 lo of a, lo of w, the dropped lo.lo term, the fp32 rounding of lrelu) + 2^-25
                              per operand element where fp16 subnormals leave an absolute half-spacing;
                   f16 + f8 : 2^-13 |a||w| (E4M3 half-ulp 2^-4 on a_lo, on w_hi, and on both factors of a_hi.w_lo, each of those terms
                              <= 2^-11 |a||w|; the header's ~2^-16 is the typical, not the worst, size) + 2^-20 |w| per activation
                              element and 2^-21 max|w| |a| for the E4M3 subnormal range;
      saturated  outputs whose inputs include an activation beyond the split's range (fp16: 65504, f16 + f8: 256): op_bound does not
                 hold there, only the contract does."""
    taps, cin, n = w.shape
    if segments:
        segs = [(tap, kc) for tap in range(taps) for kc in range(cin // 256)]
    else:
        segs = [None]
    contract = 0.0
    acc = 0.0
    for seg in segs:
        ws = w
        if seg is not None:
            tap, kc = seg
            ws = torch.zeros_like(w)
            ws[tap, kc * 256:(kc + 1) * 256] = w[tap, kc * 256:(kc + 1) * 256]
        a, parts, s = _split_operands(x, ws, in_act, in_slope, f8)
        c = sum(lin(p, q, dil, pad) for p, q in parts) / s
        mag = sum(lin(p.abs(), q.abs(), dil, pad) for p, q in parts) / s
        n_mma = (2 if f8 else 3) * (1 if seg is not None else taps) * ((256 if seg is not None else cin) // 16)
        contract = contract + c
        acc = acc + n_mma * 2.0 ** -23 * mag + (U * (contract.abs() + mag) if seg is not None else 0.0)
    aa, wa = a.abs(), w.double().abs()
    ones_a, ones_w = torch.ones_like(aa), torch.ones_like(wa)
    if f8:
        op = 2.0 ** -13 * lin(aa, wa, dil, pad) + 2.0 ** -20 * lin(ones_a, wa, dil, pad) + 2.0 ** -21 * wa.max() * lin(aa, ones_w, dil, pad)
    else:
        s = packing.split_fp16(w)[2]
        op = 4 * 2.0 ** -22 * lin(aa, wa, dil, pad) + 2.0 ** -25 * (lin(ones_a, wa, dil, pad) + lin(aa, ones_w, dil, pad) / s)
    sat = lin((aa > (F8_SAT if f8 else F16_MAX)).double(), ones_w[..., :1], dil, pad)[..., :1] > 0
    return contract, acc, op, sat


def epilogue_bound(pre, bias, res, y0):
    """fp32 epilogue: bias add, activation, residual add, alpha, accumulate add -- a few roundings of at most u each of the operands."""
    t = pre.abs()
    for v in (bias, res, y0):
        if v is not None:
            t = t + v.double().abs()
    return 8 * U * t


# ------------------------------------------------------------------------------------------------ a. attention, peaked softmax
ATT_T, ATT_H, ATT_DH = 300, 2, 128
ATT_LENS = [1, 63, 64, 65, 127, 128, 129, 300]          # 64-key (fp32 kernel) and 128-key (tensor-core kernels) block edges


def _attention_case(kind, seed=0):
    """qkv [B,T,3*H*Dh] for one softmax regime; returns (qkv, lens)."""
    B, T, H, Dh = len(ATT_LENS), ATT_T, ATT_H, ATT_DH
    gen = g(seed)
    q = torch.randn(B, T, H, Dh, generator=gen)
    k = torch.randn(B, T, H, Dh, generator=gen)
    v = torch.randn(B, T, H, Dh, generator=gen)
    if kind.startswith("peaked"):                       # logit std = sigma_q * sigma_k * sqrt(Dh) * Dh^-0.5
        sd = math.sqrt(float(kind[6:]))
        q, k = q * sd, k * sd
    elif kind == "masked_max":                          # padded rows huge: the largest logit of every padded row sits in a masked key
        q, k = q * 2.0, k * 2.0
        for b, n in enumerate(ATT_LENS):
            for t_ in (q, k, v):
                t_[b, n:] = 1.0e3 * torch.sign(torch.randn(T - n, H, Dh, generator=gen))
    elif kind == "very_negative":                       # every valid logit ~ -200: exp underflows without the maximum subtraction
        c = math.sqrt(200.0 / math.sqrt(Dh))
        q, k = c + 0.5 * q, -c + 0.5 * k
    elif kind == "jump":                                # row maximum moves by 120 between 64-key blocks: 0, +120, +240, 0, +120
        off = torch.tensor([(s // 64) % 3 for s in range(T)], dtype=torch.float32) * (120.0 / (2.0 * math.sqrt(Dh)))
        q = 2.0 + 0.5 * q
        k = 0.5 * k + off[None, :, None, None]
    qkv = torch.cat([t_.reshape(B, T, H * Dh) for t_ in (q, k, v)], dim=-1).contiguous()
    return qkv, torch.tensor(ATT_LENS, dtype=torch.int32)


def attention_bound(qkv, lens, split):
    """Per-element bound on |ctx - exact| for one backend, from the operand / accumulator model (first order):
      logit error  d_s = scale * sum_j (e(q_j)|k_j| + |q_j| e(k_j)) + acc * A_s,   A_s = scale * sum_j |q_j k_j|
                   fp32 kernel:  e = 0, acc = (Dh + 4) u   (Dh-term fp32 dot product, the scale multiply, the max subtraction)
                   split-fp16:   e(x) = 2^-22 |x| + 2^-24 (fp16 lo, subnormal spacing), acc = 24 * 2^-23 (3 MMAs x 8 K-steps) + 4u
                   plus 2^-22 for expf / ex2.approx, counted as a logit error;
      softmax      |dp_s| <= 2 max_s d_s * p_s, so the ctx error is <= 2 max_s d_s * max_s |v_s|;
      P.V          fp32: (n + 4) u sum_s p_s|v_s| plus 2^-23 per online-rescale block of 64 keys;
                   split: sum_s (2^-22 p_s + 2^-24)|v_s| + 2^-22 p_s|v_s| (p hi/lo planes, V tiles) + 3 * ceil(n / 16) 2^-23 sum_s p_s|v_s|;
      + 2^-23 |ctx| for the final normalisation.  Padded query rows are exact zeros (contract)."""
    B, T, D3 = qkv.shape
    D = D3 // 3
    Dh = ATT_DH
    x = qkv.double()
    q, k, v = (x[..., i * D:(i + 1) * D].reshape(B, T, ATT_H, Dh).permute(0, 2, 1, 3) for i in range(3))
    scale = Dh ** -0.5
    key_ok = (torch.arange(T)[None, :] < lens[:, None].long())[:, None, None, :]        # [B,1,1,T]
    s = (q @ k.transpose(-1, -2)) * scale
    p = torch.softmax(s.masked_fill(~key_ok, float("-inf")), -1)
    ctx = p @ v
    A = (q.abs() @ k.abs().transpose(-1, -2)) * scale
    if split:
        eq, ek = 2.0 ** -22 * q.abs() + U, 2.0 ** -22 * k.abs() + U
        dl = scale * (eq @ k.abs().transpose(-1, -2) + q.abs() @ ek.transpose(-1, -2)) + (24 * 2.0 ** -23 + 4 * U) * A
    else:
        dl = (Dh + 4) * U * A
    dl = (dl + 2.0 ** -22).masked_fill(~key_ok, 0.0).amax(-1, keepdim=True)               # [B,H,T,1]
    vmask = key_ok.transpose(-1, -2).double()                                             # [B,1,T,1]
    vmax = (v.abs() * vmask).amax(-2, keepdim=True)                                       # [B,H,1,Dh]
    pv = p @ v.abs()
    n = lens.double()[:, None, None, None]
    if split:
        pv_err = (p * 2.0 ** -22) @ v.abs() + U * (v.abs() * vmask).sum(-2, keepdim=True) + 2.0 ** -22 * pv \
            + 3 * torch.ceil(n / 16) * 2.0 ** -23 * pv
    else:
        pv_err = (n + 4) * U * pv + (torch.ceil(n / 64) + 1) * 2.0 ** -23 * pv
    bound = 2 * dl * vmax + pv_err + 2.0 ** -23 * ctx.abs()
    to_btd = lambda t: t.permute(0, 2, 1, 3).reshape(B, T, D)
    row_ok = (torch.arange(T)[None, :] < lens[:, None].long())[..., None]
    return to_btd(ctx).masked_fill(~row_ok, 0.0), to_btd(bound), s, key_ok


@pytest.mark.parametrize("backend", [0, 1, 2])
@pytest.mark.parametrize("kind", ["peaked4", "peaked16", "peaked40", "masked_max", "very_negative", "jump"])
def test_attention_value_ranges(kind, backend, parity_log):
    """fs2_attention where the softmax's maximum subtraction matters (all three ways the backends find it: online rescale in the fp32
    kernel, per-row registers in the GEMM path's softmax, two passes in the fused kernel).  Each case checks its own premise, then the
    output against fp64 with the bound of attention_bound(); padded query rows must be exact zeros and every output finite."""
    qkv, lens = _attention_case(kind)
    want, bound, s, key_ok = attention_bound(qkv, lens, split=backend != 0)
    smax_valid = s.masked_fill(~key_ok, float("-inf")).amax(-1)                          # [B,H,T]
    if kind == "masked_max":
        pad = torch.tensor([n < ATT_T for n in ATT_LENS])
        assert (s.amax(-1)[pad] > smax_valid[pad] + 100).all()
    if kind == "very_negative":
        assert (smax_valid < -150).all()
    if kind == "jump":
        d = s[..., 64:128].amax(-1) - s[..., :64].amax(-1)
        assert (d[lens.long() > 64] > 100).all()
    got = ops.attention(qkv.to(DEV), ATT_H, lens.to(DEV), backend=backend).cpu()
    torch.cuda.synchronize()
    assert torch.isfinite(got).all()
    for b, n in enumerate(ATT_LENS):
        assert (got[b, n:] == 0).all()
    err = (got.double() - want).abs()
    ratio = (err / bound).max().item()
    err32 = (E.attention(qkv, ATT_H, lens).double() - want).abs().max().item()      # the same contract evaluated in fp32 (torch, CPU)
    parity_log(f"attention_range_{kind}_backend{backend}", max_abs_err=err.max().item(), max_err_over_bound=ratio, cpu_fp32_max_abs_err=err32)
    assert ratio <= 1.0, (err.max().item(), ratio)
    # the bound above is a worst case; the kernel must also stay at the fp32 level (the fuzzy-model pattern of
    # test_gpu_ops.py::test_conv1d_tensor_core_k_segmented: within 4x of an fp32 evaluation's own error)
    assert err.max().item() <= 4 * err32 + 2 * U, (err.max().item(), err32)


# ------------------------------------------------------------------------------------------------ b. split-operand convs across magnitudes
RANGE_TC_CASES = [
    # B, T, Cin, N, taps, dil, pad, in_act, out_act, res, alpha, accumulate      (a subset of test_gpu_ops.py::TC_CASES)
    (1, 128, 16, 128, 1, 1, 0, 0, 0, False, 1.0, False),      # one tile, one K-block
    (2, 700, 128, 128, 11, 5, 25, 3, 3, True, 1.0, False),    # HiFi-GAN stage-1 conv1: dilation 5, lrelu in/out
    (2, 333, 512, 80, 5, 1, 2, 0, 0, True, 1.0, False),       # PostNet last conv, N = 80
    (2, 1500, 32, 32, 3, 3, 3, 3, 3, False, 1.0, False),      # 32 channels, MT = 4
    (2, 257, 64, 64, 2, 1, 1, 3, 0, False, 1.0, True),        # ConvTranspose phase group, accumulate
]


def _scaled_x(B, T, Cin, scale, seed):
    """randn activations with a per-row scale of scale * {1/2, 1, 2} (rows cycle), so every case straddles its nominal magnitude."""
    row = scale * torch.tensor([0.5, 1.0, 2.0])[torch.arange(T) % 3]
    return rnd(B, T, Cin, seed=seed) * row[None, :, None]


@pytest.mark.parametrize("f8", [False, True])
@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("case", RANGE_TC_CASES)
def test_conv1d_tensor_core_value_ranges(case, scale, f8, parity_log):
    """fs2_conv1d on the tensor cores (three-MMA split and FS2_TC_VARIANT_F8) with activations from 1e-5 to 3e4:
      (a) contract, tight: against the exactly rounded operands of _split_operands (fp16 saturation, E4M3 saturation and subnormals
          included) the only difference allowed is the accumulator and the epilogue: acc_bound + epilogue_bound of tc_model -- so the
          kernel saturates exactly where the packer and the emulation say, with no NaN and no wrong byte;
      (b) against the exact fp64 result: op_bound of tc_model on top, asserted only for outputs whose inputs stay below the split's
          saturation point (fp16 65504, f16 + f8 256); beyond it the error is logged."""
    B, T, Cin, N, taps, dil, pad, in_act, out_act, use_res, alpha, acc = case
    x = _scaled_x(B, T, Cin, scale, seed=1)
    w = rnd(taps, Cin, N, seed=2, scale=(taps * Cin) ** -0.5)
    bias = rnd(N, seed=3, scale=0.1)
    res = rnd(B, T, N, seed=4) if use_res else None
    y0 = rnd(B, T, N, seed=5) if acc else None
    d = lambda t: None if t is None else t.double()
    pre, acc_b, op_b, sat = tc_model(x, w, dil=dil, pad=pad, in_act=in_act, in_slope=0.1, f8=f8)
    exact_pre = lin(E._act(x.double(), in_act, 0.1), w.double(), dil, pad)
    want = E.conv1d_epilogue(pre, bias.double(), out_act, 0.1, d(res), alpha, d(y0))
    exact = E.conv1d_epilogue(exact_pre, bias.double(), out_act, 0.1, d(res), alpha, d(y0))
    wtc = packing.pack_conv_tc(w, f8=f8)
    out = y0.to(DEV).clone() if acc else None
    got = ops.conv1d(x.to(DEV), w.to(DEV), bias.to(DEV), dilation=dil, pad_left=pad, in_act=in_act, in_slope=0.1, out_act=out_act,
                     out_slope=0.1, res=None if res is None else res.to(DEV), alpha=alpha, out=out, accumulate=acc,
                     w_tc=wtc.to(DEV), backend=2, tc_variant=int(f8)).cpu().double()
    assert torch.isfinite(got).all()
    b_contract = acc_b + epilogue_bound(pre, bias, res, y0)
    r_contract = ((got - want).abs() / b_contract).max().item()
    ok = ~sat.expand_as(got)
    e_exact = (got - exact).abs()
    r_exact = (e_exact / (b_contract + op_b))[ok].max().item() if ok.any() else float("nan")
    parity_log(f"conv_tc_range_{'f8' if f8 else 'split3'}_{Cin}x{N}k{taps}_s{scale:g}", contract_over_bound=r_contract,
               exact_over_bound_unsaturated=r_exact, exact_max_abs_err=e_exact.max().item(), saturated_fraction=(~ok).double().mean().item(),
               max_abs_out=exact.abs().max().item())
    assert r_contract <= 1.0, r_contract
    assert not ok.any() or r_exact <= 1.0, r_exact


RANGE_SEG_CASES = [
    # B, T, Cin, N, taps, pad, in_act, res      (test_gpu_ops.py::SEG_CASES without the row mask)
    (2, 128, 256, 768, 1, 0, 0, False),
    (3, 100, 256, 1024, 9, 4, 0, False),
    (2, 128, 1024, 256, 1, 0, 3, True),
]


@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("case", RANGE_SEG_CASES)
def test_conv1d_tensor_core_k_segmented_value_ranges(case, scale, parity_log):
    """FS2_TC_VARIANT_NB64 | SEGMENTED (every (tap, 256-channel) segment with its own weight scale and a fresh accumulator) across the
    same magnitudes, with the same two checks as test_conv1d_tensor_core_value_ranges (tc_model with segments=True).  The segments add
    into y in fp32 and the bias goes in with the first, so each of the taps * Cin / 256 adds may round away u of |bias| as well."""
    B, T, Cin, N, taps, pad, in_act, use_res = case
    x = _scaled_x(B, T, Cin, scale, seed=1)
    w = rnd(taps, Cin, N, seed=2, scale=(taps * Cin) ** -0.5)
    bias = rnd(N, seed=3, scale=0.1)
    res = rnd(B, T, N, seed=4) if use_res else None
    d = lambda t: None if t is None else t.double()
    pre, acc_b, op_b, sat = tc_model(x, w, pad=pad, in_act=in_act, in_slope=0.0, segments=True)
    exact_pre = lin(E._act(x.double(), in_act, 0.0), w.double(), 1, pad)
    want = E.conv1d_epilogue(pre, bias.double(), 0, 0.0, d(res))
    exact = E.conv1d_epilogue(exact_pre, bias.double(), 0, 0.0, d(res))
    wseg = packing.pack_conv_tc_segments(w)
    got = ops.conv1d(x.to(DEV), w.to(DEV), bias.to(DEV), pad_left=pad, in_act=in_act, in_slope=0.0, res=None if res is None else res.to(DEV),
                     w_tc=wseg.to(DEV), backend=2, tc_variant=2 | 4).cpu().double()
    assert torch.isfinite(got).all()
    n_seg = taps * Cin // 256
    b_contract = acc_b + epilogue_bound(pre, bias, res, None) + n_seg * U * bias.double().abs()    # every segment's add carries the bias
    r_contract = ((got - want).abs() / b_contract).max().item()
    ok = ~sat.expand_as(got)
    e_exact = (got - exact).abs()
    r_exact = (e_exact / (b_contract + op_b))[ok].max().item() if ok.any() else float("nan")
    parity_log(f"conv_tc_seg_range_{Cin}x{N}k{taps}_s{scale:g}", contract_over_bound=r_contract, exact_over_bound_unsaturated=r_exact,
               exact_max_abs_err=e_exact.max().item(), saturated_fraction=(~ok).double().mean().item())
    assert r_contract <= 1.0, r_contract
    assert not ok.any() or r_exact <= 1.0, r_exact


def _resblock_weights(C, k, seed):
    return rnd(C, C, k, seed=seed, scale=0.6 * (C * k) ** -0.5), rnd(C, seed=seed + 1000, scale=0.05)


@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("mode", ["group", "pair"])
def test_resstack_value_ranges(mode, scale, parity_log):
    """fs2_resstack across the magnitudes, in group mode (three kernel sizes, mean) and in single-pair mode (alpha, accumulate).  Its
    layers use the per-layer kernel's f16 + f8 operands, so the reference for its error is that of the same chain run layer by layer
    through fs2_conv1d (FS2_TC_VARIANT_F8, the vocoder's unfused path) against fp64: the fused kernel must stay within 4x of it (the
    fuzzy-model pattern of test_conv1d_tensor_core_k_segmented; only summation order and on-chip intermediates differ), and finite."""
    B = 2
    if mode == "group":
        N, C, kernels, dils, alpha, accumulate = 700, 32, (3, 7, 11), ((1, 3, 5),) * 3, 0.0, False
    else:
        N, C, kernels, dils, alpha, accumulate = 1000, 64, (3,), ((5,),), 1.0 / 3, True
    x = _scaled_x(B, N, C, scale, seed=21)
    y0 = rnd(B, N, C, seed=22) if accumulate else None
    nk = len(kernels)
    w1, b1, w2, b2 = [], [], [], []
    want = torch.zeros(B, N, C, dtype=torch.float64)
    layered = torch.zeros(B, N, C, device=DEV)
    xd = x.to(DEV)
    for j, k in enumerate(kernels):
        w1.append([]); b1.append([]); w2.append([]); b2.append([])
        r = x.double().transpose(1, 2)
        rl = xd
        for di, dv in enumerate(dils[j]):
            wa, ba = _resblock_weights(C, k, 100 + 10 * j + di)
            wb, bb = _resblock_weights(C, k, 200 + 10 * j + di)
            t = F.conv1d(F.leaky_relu(r, 0.1), wa.double(), ba.double(), dilation=dv, padding=(k - 1) * dv // 2)
            r = F.conv1d(F.leaky_relu(t, 0.1), wb.double(), bb.double(), padding=(k - 1) // 2) + r
            ta = packing.pack_conv_tc(packing.conv_w(wa), f8=True).to(DEV)
            tb = packing.pack_conv_tc(packing.conv_w(wb), f8=True).to(DEV)
            w1[j].append(ta); b1[j].append(ba.to(DEV)); w2[j].append(tb); b2[j].append(bb.to(DEV))
            tl = ops.conv1d(rl, packing.conv_w(wa).to(DEV), ba.to(DEV), dilation=dv, pad_left=(k - 1) * dv // 2, in_act=3, in_slope=0.1,
                            w_tc=ta, backend=2, tc_variant=1)
            rl = ops.conv1d(tl, packing.conv_w(wb).to(DEV), bb.to(DEV), pad_left=(k - 1) // 2, in_act=3, in_slope=0.1, res=rl,
                            w_tc=tb, backend=2, tc_variant=1)
        want += r.transpose(1, 2)
        layered += rl
    a_eff = alpha if alpha > 0 else 1.0 / nk
    want = want * a_eff + (y0.double() if accumulate else 0.0)
    layered = layered * a_eff + (y0.to(DEV) if accumulate else 0.0)
    out = y0.to(DEV).clone() if accumulate else None
    got = ops.resstack(xd, kernels, dils, w1, b1, w2, b2, alpha=alpha, out=out, accumulate=accumulate)
    torch.cuda.synchronize()
    assert torch.isfinite(got).all()
    err = (got.cpu().double() - want).abs().max().item()
    err_layered = (layered.cpu().double() - want).abs().max().item()
    floor = 2 * U * want.abs().max().item()
    parity_log(f"resstack_range_{mode}_s{scale:g}", max_abs_err=err, layered_max_abs_err=err_layered, max_abs_out=want.abs().max().item())
    assert err <= 4 * err_layered + floor, (err, err_layered)


# ------------------------------------------------------------------------------------------------ c. strided / offset tensor-core outputs
SENTINEL = -12345.0


@pytest.mark.parametrize("f8", [False, True])
@pytest.mark.parametrize("u,cin,cout", [(8, 512, 256), (8, 256, 128), (2, 128, 64), (2, 64, 32)])
def test_conv_transpose_phase_groups_tensor_core(u, cin, cout, f8, parity_log):
    """Both ConvTranspose1d phase groups of one HiFi-GAN stage through the tcgen05 kernel, written as vocoder_impl writes them: one
    [B, T, u*C_out] buffer, y_row_stride = u*C_out, y and bias offset by g*(u/2)*C_out.  The buffer (with guard elements on both sides) is
    pre-filled with a sentinel: group A must leave group B's columns untouched and neither may write outside the buffer.  Result against
    fp64 conv_transpose1d with tc_model's bound (contract tight; exact bound where no activation saturates)."""
    B, T = 2, 37
    w = rnd(cin, cout, 2 * u, seed=7, scale=(2 * cin) ** -0.5)
    x = rnd(B, T, cin, seed=8)
    bias = rnd(cout, seed=9, scale=0.1)
    half = u // 2
    wa, wb = packing.split_conv_transpose(w, u)
    bt = bias.repeat(u)
    guard = 64
    flat = torch.full((B * T * u * cout + 2 * guard,), SENTINEL, device=DEV)
    out = flat[guard:guard + B * T * u * cout].view(B, T, u * cout)
    xd = x.to(DEV)
    want_parts, bound_parts = [], []
    for gi, (wg, padl) in enumerate(((wa, 1), (wb, 0))):
        cols = slice(gi * half * cout, (gi + 1) * half * cout)
        ops.conv1d(xd, wg.to(DEV), bt[cols].contiguous().to(DEV), pad_left=padl, in_act=3, in_slope=0.1, out=out[:, :, cols],
                   w_tc=packing.pack_conv_tc(wg, f8=f8).to(DEV), backend=2, tc_variant=int(f8))
        torch.cuda.synchronize()
        if gi == 0:
            assert (out[:, :, half * cout:] == SENTINEL).all()
        pre, acc_b, op_b, sat = tc_model(x, wg, pad=padl, in_act=3, in_slope=0.1, f8=f8)
        assert not sat.any()
        want_parts.append(pre + bt[cols].double())
        bound_parts.append(acc_b + op_b + epilogue_bound(pre, bt[cols], None, None))
    assert (flat[:guard] == SENTINEL).all() and (flat[-guard:] == SENTINEL).all()
    got = out.cpu().double()
    contract = torch.cat(want_parts, -1)
    exact = F.conv_transpose1d(F.leaky_relu(x.double(), 0.1).transpose(1, 2), w.double(), bias.double(), stride=u,
                               padding=u // 2).transpose(1, 2).reshape(B, T, u * cout)
    bound = torch.cat(bound_parts, -1)
    r_contract = ((got - contract).abs() / bound).max().item()
    r_exact = ((got - exact).abs() / bound).max().item()
    parity_log(f"conv_transpose_tc_u{u}_{cin}x{cout}_{'f8' if f8 else 'split3'}", exact_max_abs_err=(got - exact).abs().max().item(),
               exact_over_bound=r_exact, contract_over_bound=r_contract)
    assert r_contract <= 1.0 and r_exact <= 1.0, (r_contract, r_exact)


@pytest.mark.parametrize("f8", [False, True])
def test_conv_pre_strided_mel_view(f8, parity_log):
    """conv_pre (80 -> 512, k = 7) reading a channels-last mel VIEW with row stride 96 floats (32-byte aligned, strides % 8 == 0) through
    FS2_CONV_TC; then the same view moved by 16 bytes: FS2_CONV_TC refuses it and FS2_CONV_AUTO serves it with the exact fp32 kernel,
    whose bound is (K + 2) u sum|x||w| (K = 560 products, bias) plus the output rounding."""
    from fastspeech2_b200._lib import Fs2Error
    B, T, C, N, taps = 2, 150, 80, 512, 7
    mel = (rnd(B, T, 96, seed=31) * 2.0 - 5.0).clamp(-11.5, 2.0)      # log-mel range, as synth.make_mels
    w = rnd(taps, C, N, seed=32, scale=(taps * C) ** -0.5)
    bias = rnd(N, seed=33, scale=0.1)
    buf = torch.zeros(B * T * 96 + 8, device=DEV)
    aligned = buf[:B * T * 96].view(B, T, 96)
    aligned.copy_(mel.to(DEV))
    xv = aligned[:, :, :C]
    assert xv.data_ptr() % 32 == 0 and xv.stride(1) == 96
    x = mel[:, :, :C]
    pre, acc_b, op_b, sat = tc_model(x, w, pad=3, f8=f8)
    assert not sat.any()
    exact = lin(x.double(), w.double(), 1, 3) + bias.double()
    got = ops.conv1d(xv, w.to(DEV), bias.to(DEV), pad_left=3, w_tc=packing.pack_conv_tc(w, f8=f8).to(DEV), backend=2,
                     tc_variant=int(f8)).cpu().double()
    bound = acc_b + op_b + epilogue_bound(pre, bias, None, None)
    r_contract = ((got - (pre + bias.double())).abs() / bound).max().item()
    r_exact = ((got - exact).abs() / bound).max().item()
    assert r_contract <= 1.0 and r_exact <= 1.0, (r_contract, r_exact)
    mis = buf[4:4 + B * T * 96].view(B, T, 96)
    mis.copy_(mel.to(DEV))
    xm = mis[:, :, :C]
    assert xm.data_ptr() % 32 == 16
    wtc = packing.pack_conv_tc(w, f8=f8).to(DEV)
    with pytest.raises(Fs2Error):
        ops.conv1d(xm, w.to(DEV), bias.to(DEV), pad_left=3, w_tc=wtc, backend=2, tc_variant=int(f8))
    got_auto = ops.conv1d(xm, w.to(DEV), bias.to(DEV), pad_left=3, w_tc=wtc, backend=0, tc_variant=int(f8)).cpu().double()
    b32 = (taps * C + 2) * U * (lin(x.double().abs(), w.double().abs(), 1, 3) + bias.double().abs()) + U * exact.abs()
    r_auto = ((got_auto - exact).abs() / b32).max().item()
    parity_log(f"conv_pre_strided_{'f8' if f8 else 'split3'}", tc_exact_over_bound=r_exact, tc_contract_over_bound=r_contract,
               auto_misaligned_over_fp32_bound=r_auto)
    assert r_auto <= 1.0, r_auto


# ------------------------------------------------------------------------------------------------ d. row ops
@pytest.mark.parametrize("C", [256, 80])
def test_layernorm_pre_relu(C, parity_log):
    """fs2_layernorm with pre_relu = 1 (LayerNorm(relu(x)), the predictors' conv -> ReLU -> LayerNorm) on random rows, all-negative rows
    (relu gives a zero row: variance 0, output = beta exactly) and rows with a mean of 100x their spread, with and without row_lens.
    Bar: the fp32 two-pass statistics -- the mean's error <= 16 u mean|v| (4-wide pairwise, 8 per lane, 5 shuffle levels), which shifts
    every output by <= that * rstd * |gamma|; the variance sum (16 u, i.e. 8 u in rstd), rsqrtf (2 ulp) and the subtract / scale / shift
    roundings add <= 16 u of |y| and |beta|."""
    B, T = 3, 40
    x = rnd(B, T, C, seed=1, scale=3.0)
    x[0, 5:9] = -x[0, 5:9].abs() - 0.1                            # all-negative rows
    x[1, :20] = 100.0 + rnd(20, C, seed=2, scale=1.0)             # mean offset 100 x std
    gm, bt = 1 + rnd(C, seed=3, scale=0.1), rnd(C, seed=4, scale=0.1)
    lens = torch.tensor([T, 13, 1], dtype=torch.int32)
    v = torch.relu(x).double()
    mean = v.mean(-1, keepdim=True)
    var = v.var(-1, unbiased=False, keepdim=True)
    rstd = (var + 1e-5).rsqrt()
    yhat = (v - mean) * rstd
    bound = 16 * U * v.abs().mean(-1, keepdim=True) * rstd * gm.double().abs() + 16 * U * ((yhat * gm.double()).abs() + bt.double().abs())
    for ln_ in (None, lens):
        want = E.layernorm(v, gm.double(), bt.double(), ln_)
        got = ops.layernorm(x.to(DEV), gm.to(DEV), bt.to(DEV), None if ln_ is None else ln_.to(DEV), pre_relu=True).cpu().double()
        assert torch.equal(got[0, 5:9].float(), bt.expand(4, C))      # variance 0: exactly beta
        if ln_ is not None:
            for b, n in enumerate(lens.tolist()):
                assert (got[b, n:] == 0).all()
        ratio = ((got - want).abs() / bound).max().item()
        parity_log(f"layernorm_pre_relu_C{C}_{'lens' if ln_ is not None else 'nolens'}", max_abs_err=(got - want).abs().max().item(),
                   max_err_over_bound=ratio)
        assert ratio <= 1.0, ratio


def test_add_positions():
    """fs2_add_positions: x[b,t,:] += pos[t,:] -- one fp32 add per element, bit exact; pos rows beyond T are not read."""
    B, T, D = 3, 77, 256
    x = rnd(B, T, D, seed=1)
    pos = rnd(T + 5, D, seed=2)
    xd = x.to(DEV)
    L.check(L.lib().fs2_add_positions(xd.data_ptr(), pos.to(DEV).data_ptr(), B, T, D, torch.cuda.current_stream().cuda_stream),
            "fs2_add_positions")
    torch.cuda.synchronize()
    assert torch.equal(xd.cpu(), x + pos[:T])


def test_durations_non_finite_and_targets():
    """fs2_durations edge cases.  Predicted log-durations giving NaN, +inf (exp overflow) or more than 1e6 frames are counted in
    len_stats[2] and contribute 0 frames to cum and mel_lens (the reference raises on them; the caller can fail loudly); d_rounded keeps
    torch.clamp's NaN.  Targets: negative values give 0 frames (max((int)d, 0)) and d_control is ignored."""
    B, Lp = 3, 300
    logd = rnd(B, Lp, seed=1, scale=0.6) + 1.2
    logd[0, 3] = float("nan")
    logd[0, 10] = 100.0                                  # exp -> inf
    logd[1, 7] = 14.5                                    # ~2.0e6 frames
    logd[1, 299] = float("inf")
    logd[2, 0] = float("-inf")                           # exp -> 0 -> rint(-1) -> clamp -> 0 frames, not wild
    d, cum, mel_lens, mel_lens32, stats = ops.durations(logd.to(DEV), False, 1.0)
    want_d = torch.clamp(torch.round(torch.exp(logd) - 1) * 1.0, min=0)
    wild = ~(want_d <= 1e6)
    reps = torch.where(wild, torch.zeros_like(want_d), want_d).to(torch.int32)
    want_cum = torch.cumsum(reps, 1).to(torch.int32)
    assert int(wild.sum()) == 4
    d = d.cpu()
    assert torch.equal(d.isnan(), want_d.isnan()) and torch.equal(d.nan_to_num(), want_d.nan_to_num())
    assert torch.equal(cum.cpu(), want_cum) and torch.equal(mel_lens.cpu(), want_cum[:, -1].long())
    assert torch.equal(mel_lens32.cpu(), want_cum[:, -1])
    assert stats.cpu().tolist() == [int(want_cum[:, -1].max()), int(want_cum[:, -1].sum()), 4]
    tgt = torch.randint(-3, 9, (B, Lp), generator=g(4)).float()
    tgt[2, 5] = -0.5
    _, wcum, wlen = E.durations(tgt, True, 1.0)
    for dc in (1.0, 2.5):
        _, cum2, ml2, _, st2 = ops.durations(tgt.to(DEV), True, dc)
        assert torch.equal(cum2.cpu(), wcum) and torch.equal(ml2.cpu(), wlen)
        assert st2.cpu().tolist() == [int(wlen.max()), int(wlen.sum()), 0]


def test_embed_and_speaker_out_of_range_ids():
    """fs2_embed_positions / fs2_add_speaker with ids < 0 and >= the table size read row 0 (rowwise.cu: the reference would raise; the
    kernels stay in bounds).  This pins that rule."""
    n_vocab, D = 50, 256
    table = rnd(n_vocab, D, seed=1)
    pos = rnd(40, D, seed=2)
    ids = torch.randint(0, n_vocab, (3, 17), generator=g(3))
    ids[0, 0], ids[0, 5], ids[1, 16], ids[2, 3] = -1, n_vocab, n_vocab + 1000, -(2 ** 40)
    y = ops.embed_positions(ids.to(DEV), table.to(DEV), pos.to(DEV)).cpu()
    safe = torch.where((ids < 0) | (ids >= n_vocab), torch.zeros_like(ids), ids)
    assert torch.equal(y, table[safe] + pos[:17])
    spk = rnd(4, D, seed=4)
    sid = torch.tensor([-2, 4, 3])
    y2 = ops.add_speaker_(y.to(DEV), spk.to(DEV), sid.to(DEV)).cpu()
    assert torch.equal(y2, y + spk[torch.tensor([0, 0, 3])][:, None, :])


def _np_int16(wav, scale, lens):
    """The reference's host conversion, utils/model.py:82-90: (wav * max_wav_value).astype("int16"), then wav[i][:lengths[i]]
    (here: samples t >= lens[b] are 0, as fs2_wav_to_int16 writes them)."""
    with np.errstate(invalid="ignore"):
        out = (wav.numpy() * scale).astype("int16")
    if lens is not None:
        for b, n in enumerate(lens):
            out[b, max(n, 0):] = 0
    return out


SPECIAL = [1.0, -1.0, float(np.nextafter(np.float32(1), np.float32(0))), -float(np.nextafter(np.float32(1), np.float32(0))), 1.5, 2.0,
           70000 / 32768, -70000 / 32768, 65537 / 32768, 1e5, -1e5, float("nan"), float("inf"), float("-inf"), 0.5 / 32768, -1.5 / 32768, 0.0]


@pytest.mark.parametrize("N,lens,strided", [(1003, None, False), (1003, [0, -5, 2000, 517], False), (4096, [4096, 1, 8, 4095], False),
                                            (1003, [1003, 999, 7, 1], True), (24, None, True)])
def test_wav_to_int16_matches_numpy_cast(N, lens, strided):
    """fs2_wav_to_int16 against numpy's own cast of the same samples: N not a multiple of 8, a batch stride that breaks the 16-byte path,
    lens NULL / 0 / negative / > N, and the values where a clamp and numpy differ: exactly +-1.0 (tanhf returns 1.0 for arguments
    >= ~9.01; numpy gives -32768 for +1.0), nextafter(1, 0), > 1, NaN and inf."""
    B = 4
    gen = g(5)
    base = torch.tanh(torch.randn(B, N, generator=gen) * 3.0)
    sp = torch.tensor(SPECIAL, dtype=torch.float32)
    base[0, :len(SPECIAL)] = sp                                          # head, 16-byte path
    base[1, N - len(SPECIAL):] = sp                                      # tail, scalar path when N % 8 != 0
    for b in (2, 3):
        base[b, torch.randperm(N, generator=gen)[:len(SPECIAL)]] = sp
    if strided:
        buf = torch.zeros(B, N + 3).to(DEV)
        buf[:, :N] = base.to(DEV)
        wav = buf[:, :N]
        assert wav.stride(0) % 4 != 0
    else:
        wav = base.to(DEV)
    lens_t = None if lens is None else torch.tensor(lens, dtype=torch.long)
    got = ops.wav_to_int16(wav, lens_t, 32768.0).cpu().numpy()
    want = _np_int16(base, 32768.0, lens)
    bad = np.nonzero(got != want)
    assert bad[0].size == 0, [(int(b), int(t), float(base[b, t]), int(got[b, t]), int(want[b, t])) for b, t in zip(*bad)][:10]


def test_wav_to_int16_full_scale_sample():
    """The case the reference's conversion and a clamping kernel disagree on, on its own: wav == +1.0 -> -32768 (numpy wraps 32768)."""
    wav = torch.tensor([[1.0, -1.0, 0.99999994, 2.0, float("nan"), float("inf"), 0.0, 0.5]], device=DEV)
    got = ops.wav_to_int16(wav).cpu().numpy()
    assert got.tolist() == [[-32768, -32768, 32767, 0, 0, 0, 0, 16384]]
