"""Tensor-level wrappers over the C-ABI operator entry points (include/fs2b200.h).  Plumbing only: they allocate the
output with torch and pass raw device pointers + the current stream; all arithmetic happens in libfs2b200.so."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _need_cuda(t):
    if t.device.type != "cuda":
        raise L.Fs2Error("fastspeech2_b200 ops need CUDA tensors; there is no CPU path")


def conv1d(x, w, bias=None, *, dilation=1, pad_left=0, in_act=L.ACT_NONE, in_slope=0.0, out_act=L.ACT_NONE, out_slope=0.0,
           res=None, alpha=1.0, out=None, accumulate=False, row_lens=None, w_tc=None, backend=L.CONV_AUTO, tc_variant=0):
    """x [B,T,Cin] (row-strided ok), w [taps][Cin][N] -> y [B,T,N].  `out` may be a strided [B,T,N] view."""
    _need_cuda(x)
    B, T, Cin = x.shape
    taps, _, N = w.shape
    if out is None:
        out = torch.empty(B, T, N, dtype=torch.float32, device=x.device)
    assert x.stride(2) == 1 and out.stride(2) == 1 and w.is_contiguous()
    a = L.Conv1dArgs(x=x.data_ptr(), x_batch_stride=x.stride(0), x_row_stride=x.stride(1), B=B, T=T, Cin=Cin,
                     w=w.data_ptr(), bias=L.ptr(bias), N=N, taps=taps, dilation=dilation, pad_left=pad_left,
                     w_tc=L.ptr(w_tc), backend=backend, tc_variant=tc_variant,
                     in_act=in_act, in_slope=in_slope, out_act=out_act, out_slope=out_slope,
                     res=L.ptr(res), res_batch_stride=res.stride(0) if res is not None else 0,
                     res_row_stride=res.stride(1) if res is not None else 0,
                     alpha=alpha, accumulate=int(accumulate), row_lens=L.ptr(row_lens),
                     y=out.data_ptr(), y_batch_stride=out.stride(0), y_row_stride=out.stride(1))
    L.check(L.lib().fs2_conv1d(C.byref(a), _stream(x.device)), "fs2_conv1d")
    return out


def layernorm(x, gamma, beta, row_lens=None, eps=1e-5, pre_relu=False):
    """LayerNorm over the last dim (of relu(x) with pre_relu), rows t >= row_lens[b] zeroed (fs2_layernorm)."""
    _need_cuda(x)
    B, T, Cc = x.shape
    y = torch.empty_like(x)
    a = L.LayerNormArgs(x=x.data_ptr(), y=y.data_ptr(), B=B, T=T, C=Cc, gamma=gamma.data_ptr(), beta=beta.data_ptr(), eps=eps,
                        row_lens=L.ptr(row_lens), pre_relu=int(pre_relu))
    L.check(L.lib().fs2_layernorm(C.byref(a), _stream(x.device)), "fs2_layernorm")
    return y


def attention(qkv, n_head, key_lens=None, backend=0):
    _need_cuda(qkv)
    B, T, D3 = qkv.shape
    D = D3 // 3
    ctx = torch.empty(B, T, D, dtype=torch.float32, device=qkv.device)
    ws = None
    if backend in (1, 2):
        ws = torch.empty(L.lib().fs2_attention_workspace_bytes(B, T, n_head), dtype=torch.uint8, device=qkv.device)
    a = L.AttentionArgs(qkv=qkv.data_ptr(), ctx=ctx.data_ptr(), B=B, T=T, H=n_head, Dh=D // n_head, key_lens=L.ptr(key_lens),
                        scale=float((D // n_head) ** -0.5), backend=backend, workspace=L.ptr(ws),
                        workspace_bytes=0 if ws is None else ws.numel())
    L.check(L.lib().fs2_attention(C.byref(a), _stream(qkv.device)), "fs2_attention")
    return ctx


def embed_positions(ids, table, pos):
    _need_cuda(ids)
    B, Lm = ids.shape
    y = torch.empty(B, Lm, table.shape[1], dtype=torch.float32, device=ids.device)
    a = L.EmbedArgs(ids=ids.data_ptr(), table=table.data_ptr(), pos=pos.data_ptr(), y=y.data_ptr(), B=B, L=Lm, D=table.shape[1],
                    n_vocab=table.shape[0])
    L.check(L.lib().fs2_embed_positions(C.byref(a), _stream(ids.device)), "fs2_embed_positions")
    return y


def add_speaker_(x, table, idx):
    _need_cuda(x)
    B, Lm, D = x.shape
    a = L.RowBiasArgs(x=x.data_ptr(), table=table.data_ptr(), idx=idx.data_ptr(), B=B, L=Lm, D=D, n_rows=table.shape[0])
    L.check(L.lib().fs2_add_speaker(C.byref(a), _stream(x.device)), "fs2_add_speaker")
    return x


def variance_head(h, w, b, lens=None, control=1.0, target=None, bins=None, emb=None, x=None):
    _need_cuda(h)
    B, Lm, Cc = h.shape
    pred = torch.empty(B, Lm, dtype=torch.float32, device=h.device)
    a = L.VarianceHeadArgs(h=h.data_ptr(), w=w.data_ptr(), b=b.data_ptr(), B=B, L=Lm, C=Cc, lens=L.ptr(lens), control=control,
                           target=L.ptr(target), bins=L.ptr(bins), n_edges=0 if bins is None else bins.numel(), emb=L.ptr(emb),
                           D=0 if x is None else x.shape[-1], x=L.ptr(x), pred_out=pred.data_ptr())
    L.check(L.lib().fs2_variance_head(C.byref(a), _stream(h.device)), "fs2_variance_head")
    return pred


def durations(src, use_target=False, d_control=1.0):
    _need_cuda(src)
    B, Lm = src.shape
    dev = src.device
    d_rounded = torch.empty(B, Lm, dtype=torch.float32, device=dev)
    cum = torch.empty(B, Lm, dtype=torch.int32, device=dev)
    mel_lens = torch.empty(B, dtype=torch.long, device=dev)
    mel_lens32 = torch.empty(B, dtype=torch.int32, device=dev)
    stats = torch.empty(3, dtype=torch.int32, device=dev)
    a = L.DurationsArgs(src=src.data_ptr(), use_target=int(use_target), d_control=d_control, B=B, L=Lm,
                        d_rounded=0 if use_target else d_rounded.data_ptr(), cum=cum.data_ptr(), mel_lens=mel_lens.data_ptr(),
                        mel_lens32=mel_lens32.data_ptr(), len_stats=stats.data_ptr())
    L.check(L.lib().fs2_durations(C.byref(a), _stream(dev)), "fs2_durations")
    return (None if use_target else d_rounded), cum, mel_lens, mel_lens32, stats


def length_regulate(x, cum, T, pos=None):
    _need_cuda(x)
    B, Lm, D = x.shape
    y = torch.empty(B, T, D, dtype=torch.float32, device=x.device)
    a = L.LengthRegulateArgs(x=x.data_ptr(), cum=cum.data_ptr(), pos=L.ptr(pos), y=y.data_ptr(), B=B, L=Lm, T=T, D=D)
    L.check(L.lib().fs2_length_regulate(C.byref(a), _stream(x.device)), "fs2_length_regulate")
    return y


def conv_post(x, w, bias, in_slope=0.01):
    _need_cuda(x)
    B, T, Cc = x.shape
    wav = torch.empty(B, T, dtype=torch.float32, device=x.device)
    a = L.ConvPostArgs(x=x.data_ptr(), B=B, T=T, C=Cc, w=w.data_ptr(), bias=bias.data_ptr(), taps=w.shape[0], in_slope=in_slope,
                       wav=wav.data_ptr())
    L.check(L.lib().fs2_conv_post(C.byref(a), _stream(x.device)), "fs2_conv_post")
    return wav


def resstack(x, kernels, dilations, w1_tc, b1, w2_tc, b2, alpha=0.0, out=None, accumulate=False):
    """Fused multi-receptive-field ResBlock group (fs2_resstack).  x [B,N,C] contiguous; kernels [k_j]; dilations [[d...] per j];
    w1_tc / w2_tc [j][d]: pack_conv_tc(w, f8=True) tiles; b1 / b2 [j][d]: biases."""
    _need_cuda(x)
    B, N, Cc = x.shape
    assert x.is_contiguous()
    y = torch.empty_like(x) if out is None else out
    a = L.ResstackArgs(x=x.data_ptr(), y=y.data_ptr(), B=B, N=N, C=Cc, n_kernels=len(kernels), n_dil=len(dilations[0]),
                       alpha=float(alpha), accumulate=int(accumulate))
    for j, k in enumerate(kernels):
        a.k[j] = k
        for d, dv in enumerate(dilations[j]):
            a.dil[j][d] = dv
            a.w1_tc[j][d], a.b1[j][d] = w1_tc[j][d].data_ptr(), b1[j][d].data_ptr()
            a.w2_tc[j][d], a.b2[j][d] = w2_tc[j][d].data_ptr(), b2[j][d].data_ptr()
    L.check(L.lib().fs2_resstack(C.byref(a), _stream(x.device)), "fs2_resstack")
    return y


def wav_to_int16(wav, lengths=None, scale=32768.0, out=None):
    """wav [B,N] fp32 (row-strided ok) -> int16 [B,N]: numpy's (wav*scale).astype("int16") (truncates, wraps beyond int16), samples
    t >= lengths[b] zeroed (fs2_wav_to_int16)."""
    _need_cuda(wav)
    B, N = wav.shape
    assert wav.stride(1) == 1
    if out is None:
        out = torch.empty(B, N, dtype=torch.int16, device=wav.device)
    lens = None if lengths is None else lengths.to(device=wav.device, dtype=torch.long).contiguous()
    a = L.WavInt16Args(wav=wav.data_ptr(), wav_batch_stride=wav.stride(0), B=B, N=N, lens=L.ptr(lens), scale=float(scale), out=out.data_ptr())
    L.check(L.lib().fs2_wav_to_int16(C.byref(a), _stream(wav.device)), "fs2_wav_to_int16")
    return out


def transpose_bct_to_btc(x):
    _need_cuda(x)
    B, Cc, T = x.shape
    x = x.contiguous()
    y = torch.empty(B, T, Cc, dtype=torch.float32, device=x.device)
    L.check(L.lib().fs2_transpose_bct_to_btc(x.data_ptr(), y.data_ptr(), B, Cc, T, _stream(x.device)), "fs2_transpose")
    return y
