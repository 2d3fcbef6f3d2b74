"""Thin torch-tensor wrappers over the C-ABI (lib.py): argument checking, struct filling, stream plumbing.

torch is used for device memory and streams only; every op here launches kernels of liba2f_sm100.so and raises
A2FError on any non-zero status (no fallback).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import lib as L


# bench.py's roofline pass: when set to a list, every tcgen05 GEMM launch is bracketed by CUDA events on the launch
# stream and recorded as (kind, algorithmic_flops, start_event, end_event).  None (default) = no instrumentation.
PROFILE = None


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return L.F32
    if t.dtype == torch.bfloat16:
        return L.BF16
    raise L.A2FError(f"unsupported dtype {t.dtype}")


def _dev(*ts):
    """Every tensor of a call lives on ONE CUDA device and that device is torch's current one: kernels are launched on
    torch.cuda.current_stream() of the current device with raw pointers, so a tensor of another GPU would fault (the
    drop-in modules switch devices themselves, _A2FModule.__call__; direct callers use `with torch.cuda.device(...)`)."""
    idx = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise L.A2FError("a2f ops need CUDA tensors (there is no CPU path)")
        if idx is None:
            idx = t.device.index
        elif t.device.index != idx:
            raise L.A2FError(f"a2f ops need all tensors on one device (got cuda:{idx} and cuda:{t.device.index})")
    if idx is not None and idx != torch.cuda.current_device():
        raise L.A2FError(f"tensors live on cuda:{idx} but the current device is cuda:{torch.cuda.current_device()}; "
                         f"wrap the call in `with torch.cuda.device({idx}):`")


def gemm(a: torch.Tensor, w: torch.Tensor, out: torch.Tensor, *, bias: Optional[torch.Tensor] = None,
         act: int = L.ACT_NONE, resid: Optional[torch.Tensor] = None, tmpl: Optional[torch.Tensor] = None,
         rows_per_tmpl: int = 1, backend: int = L.SIMT_F32, M: Optional[int] = None, K: Optional[int] = None,
         a_row_stride: Optional[int] = None, a_batch_stride: int = 0, rows_per_batch: Optional[int] = None,
         N: Optional[int] = None, ldw: Optional[int] = None, ldc: Optional[int] = None, c_batch_stride: int = 0,
         c_offset: int = 0, a_rows: int = 0, segs=None, resid_mode: int = 0, ldr: Optional[int] = None,
         r_batch_stride: int = 0, r_offset: int = 0, alg_K: Optional[int] = None,
         out2: Optional[torch.Tensor] = None, ldc2: Optional[int] = None) -> torch.Tensor:
    """out[m,n] = act(sum_k a[m,k] w[n,k] + bias[n]) + resid[m,n] + tmpl[m // rows_per_tmpl, n]  (a2f_gemm)."""
    _dev(a, w, out, bias, resid, tmpl)
    lib = L.load()
    g = L.GemmArgs()
    g.M = int(M if M is not None else a.shape[0])
    g.N = int(N if N is not None else w.shape[0])
    g.K = int(K if K is not None else a.shape[-1])
    g.A, g.a_dtype = a.data_ptr(), _dt(a)
    g.a_row_stride = int(a_row_stride if a_row_stride is not None else a.stride(0))
    g.a_batch_stride = int(a_batch_stride)
    g.rows_per_batch = int(rows_per_batch if rows_per_batch is not None else g.M)
    g.W, g.ldw = w.data_ptr(), int(ldw if ldw is not None else w.stride(0))
    g.bias = L.ptr(bias)
    g.act = act
    if resid is not None:
        g.resid, g.resid_dtype = resid.data_ptr() + int(r_offset) * resid.element_size(), _dt(resid)
        g.ldr = int(ldr if ldr is not None else resid.stride(0))
        g.r_batch_stride = int(r_batch_stride)
        g.resid_mode = int(resid_mode)
    g.a_rows = int(a_rows)
    if segs is not None:                       # [(row_off, col_off), ...]: explicit K segments (a2f.h)
        g.n_seg = len(segs)
        for i, (ro, co) in enumerate(segs):
            g.seg_row_off[i], g.seg_col_off[i] = int(ro), int(co)
    if tmpl is not None:
        g.tmpl, g.rows_per_tmpl = tmpl.data_ptr(), int(rows_per_tmpl)
    g.C, g.c_dtype = out.data_ptr() + int(c_offset) * out.element_size(), _dt(out)
    g.ldc = int(ldc if ldc is not None else out.stride(0))
    g.c_batch_stride = int(c_batch_stride)
    if out2 is not None:                       # out = pre-activation z, out2 = act(z) (tcgen05 pair kernel, a2f.h C2)
        _dev(out2)
        if out2.dtype != out.dtype:
            raise L.A2FError("out2 must have the dtype of out")
        g.C2, g.ldc2 = out2.data_ptr() + int(c_offset) * out2.element_size(), int(ldc2 if ldc2 is not None else g.ldc)
    if bias is not None and bias.dtype != torch.float32:
        raise L.A2FError("bias must be fp32")
    if tmpl is not None and tmpl.dtype != torch.float32:
        raise L.A2FError("tmpl must be fp32")
    if a.dtype != w.dtype:
        raise L.A2FError("A and W must share a dtype")
    if PROFILE is not None:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        L.check(lib.a2f_gemm(C.byref(g), backend, _stream()), "a2f_gemm")
        e.record()
        # alg_K: contraction length of the ALGORITHM when the operands carry an error-compensated split (bf16x3: K = 3 x alg_K)
        PROFILE.append(("gemm_tc" if backend == L.TCGEN05 else "gemm_simt", 2.0 * g.M * g.N * (alg_K if alg_K else g.K), s, e))
        return out
    L.check(lib.a2f_gemm(C.byref(g), backend, _stream()), "a2f_gemm")
    return out


def _bf16_2d(*ts):
    for t in ts:
        if t is not None and (t.dtype != torch.bfloat16 or t.dim() != 2 or t.stride(1) != 1):
            raise L.A2FError("expected 2-D bf16 operands with unit column stride")


def encoder_block(h1: torch.Tensor, w1: torch.Tensor, b1: Optional[torch.Tensor], w2: torch.Tensor, b2: Optional[torch.Tensor],
                  ln2_g: torch.Tensor, ln2_b: torch.Tensor, scratch: torch.Tensor, h_out: torch.Tensor, *,
                  att: Optional[torch.Tensor] = None, wo: Optional[torch.Tensor] = None, bo: Optional[torch.Tensor] = None,
                  h_in: Optional[torch.Tensor] = None, ln1_g: Optional[torch.Tensor] = None, ln1_b: Optional[torch.Tensor] = None,
                  wq: Optional[torch.Tensor] = None, bq: Optional[torch.Tensor] = None, qkv: Optional[torch.Tensor] = None,
                  eps: float = 1e-5) -> torch.Tensor:
    """The row-local part of a post-LN encoder layer in one tcgen05 kernel (a2f_encoder_block, include/a2f.h):
    [h1 = LN(h_in + att wo^T + bo)] -> f = gelu(h1 w1^T + b1) -> h_out = LN(h1 + f w2^T + b2) [-> qkv = h_out wq^T + bq].
    The bracketed phases run when att / wq are given."""
    _dev(h1, w1, b1, w2, b2, ln2_g, ln2_b, scratch, h_out, att, wo, bo, h_in, ln1_g, ln1_b, wq, bq, qkv)
    _bf16_2d(h1, w1, w2, scratch, h_out, att, wo, h_in, wq, qkv)
    M, N = h1.shape
    F = w1.shape[0]
    if w1.shape[1] != N or tuple(w2.shape) != (N, F) or tuple(h_out.shape) != (M, N) or scratch.shape[0] < M or scratch.shape[1] != F:
        raise L.A2FError("encoder_block: shape mismatch")
    g = L.EncoderBlockArgs()
    g.M, g.N, g.F = M, N, F
    g.h1, g.ld_h1 = h1.data_ptr(), h1.stride(0)
    g.w1, g.ld_w1, g.b1 = w1.data_ptr(), w1.stride(0), L.ptr(b1)
    g.f, g.ld_f = scratch.data_ptr(), scratch.stride(0)
    g.w2, g.ld_w2, g.b2 = w2.data_ptr(), w2.stride(0), L.ptr(b2)
    g.ln2_g, g.ln2_b = ln2_g.data_ptr(), ln2_b.data_ptr()
    g.h_out, g.ld_hout = h_out.data_ptr(), h_out.stride(0)
    g.eps = float(eps)
    flops = 4.0 * M * N * F
    if att is not None:
        if wo is None or h_in is None or ln1_g is None or ln1_b is None or tuple(att.shape) != (M, N) or \
                tuple(wo.shape) != (N, N) or tuple(h_in.shape) != (M, N):
            raise L.A2FError("encoder_block: the attention-output phase needs att, wo, h_in [M,N] and ln1")
        g.att, g.ld_att = att.data_ptr(), att.stride(0)
        g.wo, g.ld_wo, g.bo = wo.data_ptr(), wo.stride(0), L.ptr(bo)
        g.h_in, g.ld_hin = h_in.data_ptr(), h_in.stride(0)
        g.ln1_g, g.ln1_b = ln1_g.data_ptr(), ln1_b.data_ptr()
        flops += 2.0 * M * N * N
    if wq is not None:
        NQ = wq.shape[0]
        if qkv is None or wq.shape[1] != N or tuple(qkv.shape) != (M, NQ):
            raise L.A2FError("encoder_block: the in-projection phase needs wq [NQ,N] and qkv [M,NQ]")
        g.wq, g.ld_wq, g.bq, g.NQ = wq.data_ptr(), wq.stride(0), L.ptr(bq), NQ
        g.qkv, g.ld_qkv = qkv.data_ptr(), qkv.stride(0)
        flops += 2.0 * M * N * NQ
    lib = L.load()
    if PROFILE is not None:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
    L.check(lib.a2f_encoder_block(C.byref(g), _stream()), "a2f_encoder_block")
    if PROFILE is not None:
        e.record()
        PROFILE.append(("gemm_tc", flops, s, e))
    return h_out


def ffn_ln(x: torch.Tensor, w1: torch.Tensor, b1: Optional[torch.Tensor], w2: torch.Tensor, b2: Optional[torch.Tensor],
           gamma: torch.Tensor, beta: torch.Tensor, scratch: torch.Tensor, out: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """out = LayerNorm(x + gelu(x @ w1^T + b1) @ w2^T + b2) * gamma + beta: the feed-forward half of encoder_block."""
    return encoder_block(x, w1, b1, w2, b2, gamma, beta, scratch, out, eps=eps)


def gemm_ln(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], resid: torch.Tensor, gamma: torch.Tensor,
            beta: torch.Tensor, out: torch.Tensor, eps: float = 1e-5, pre_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = LayerNorm(a @ w^T + bias + resid) * gamma + beta in one tcgen05 kernel (a2f_gemm_ln): bf16 [M,K] x [N,K],
    N in {256, 512, 768}; the pre-LayerNorm sum stays in tensor memory (fp32).  pre_out (training): also store that sum as
    bf16 [M,N] for the LayerNorm backward."""
    _dev(a, w, bias, resid, gamma, beta, out, pre_out)
    for t in (a, w, resid, out) + ((pre_out,) if pre_out is not None else ()):
        if t.dtype != torch.bfloat16 or t.dim() != 2 or t.stride(1) != 1:
            raise L.A2FError("gemm_ln takes 2-D bf16 operands with unit column stride")
    M, K = a.shape
    N = w.shape[0]
    if w.shape[1] != K or tuple(resid.shape) != (M, N) or tuple(out.shape) != (M, N):
        raise L.A2FError("gemm_ln: shape mismatch")
    lib = L.load()
    if PROFILE is not None:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
    L.check(lib.a2f_gemm_ln(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), L.ptr(bias), resid.data_ptr(), resid.stride(0),
                            gamma.data_ptr(), beta.data_ptr(), float(eps), out.data_ptr(), out.stride(0), L.ptr(pre_out),
                            pre_out.stride(0) if pre_out is not None else 0, M, N, K, _stream()),
            "a2f_gemm_ln")
    if PROFILE is not None:
        e.record()
        PROFILE.append(("gemm_tc", 2.0 * M * N * K, s, e))
    return out


def gemm_wgrad(dy: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, *, backend: int, M: Optional[int] = None,
               N: Optional[int] = None, K: Optional[int] = None, dy_row_stride: Optional[int] = None,
               dy_batch_stride: int = 0, x_row_stride: Optional[int] = None, x_batch_stride: int = 0,
               rows_per_batch: Optional[int] = None, x_rows: int = 0, segs=None, ldw: Optional[int] = None,
               x_offset: int = 0, dy_offset: int = 0) -> torch.Tensor:
    """dw[n, s*K+k] += sum_m dy[m,n] * x[(b, r+roff_s), coff_s+k]   (a2f_gemm_wgrad; dw fp32, accumulated into)."""
    _dev(dy, x, dw)
    if dw.dtype != torch.float32:
        raise L.A2FError("dW must be fp32")
    if dy.dtype != x.dtype:
        raise L.A2FError("dY and X must share a dtype")
    g = L.WgradArgs()
    g.M = int(M if M is not None else dy.shape[0])
    g.N = int(N if N is not None else dy.shape[-1])
    g.K = int(K if K is not None else x.shape[-1])
    g.dtype = _dt(dy)
    g.dY = dy.data_ptr() + int(dy_offset) * dy.element_size()
    g.dy_row_stride = int(dy_row_stride if dy_row_stride is not None else dy.stride(-2))
    g.dy_batch_stride = int(dy_batch_stride)
    g.X = x.data_ptr() + int(x_offset) * x.element_size()
    g.x_row_stride = int(x_row_stride if x_row_stride is not None else x.stride(-2))
    g.x_batch_stride = int(x_batch_stride)
    g.rows_per_batch = int(rows_per_batch if rows_per_batch is not None else g.M)
    g.x_rows = int(x_rows)
    if segs is not None:
        g.n_seg = len(segs)
        for i, (ro, co) in enumerate(segs):
            g.x_row_off[i], g.x_col_off[i] = int(ro), int(co)
    g.dW, g.ldw = dw.data_ptr(), int(ldw if ldw is not None else dw.stride(0))
    lib = L.load()
    if PROFILE is not None and backend == L.TCGEN05:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        L.check(lib.a2f_gemm_wgrad(C.byref(g), backend, _stream()), "a2f_gemm_wgrad")
        e.record()
        PROFILE.append(("wgrad_tc", 2.0 * g.M * g.N * g.K * max(1, g.n_seg), s, e))
        return dw
    L.check(lib.a2f_gemm_wgrad(C.byref(g), backend, _stream()), "a2f_gemm_wgrad")
    return dw


def cast_bf16(x: torch.Tensor) -> torch.Tensor:
    _dev(x)
    x = x.contiguous()
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    L.check(L.load().a2f_cast_f32_to_bf16(x.data_ptr(), out.data_ptr(), x.numel(), _stream()), "a2f_cast_f32_to_bf16")
    return out


def voca_trunk(wptrs: "L.VocaWeights", x: torch.Tensor, one_hot: torch.Tensor, z: torch.Tensor) -> torch.Tensor:
    _dev(x, one_hot, z)
    L.check(L.load().a2f_voca_trunk(C.byref(wptrs), x.data_ptr(), one_hot.data_ptr(), one_hot.shape[1], z.data_ptr(),
                                    _dt(z), z.stride(0), x.shape[0], _stream()), "a2f_voca_trunk")
    return z


def loss_workspace(device) -> torch.Tensor:
    n = L.load().a2f_voca_loss_workspace_bytes()
    return torch.empty((n + 7) // 8, dtype=torch.float64, device=device)


def voca_loss_fwd(pred: torch.Tensor, gt: torch.Tensor, rows: int, v3: int, k_rec: float, k_vel: float,
                  ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    _dev(pred, gt)
    out3 = torch.empty(3, dtype=torch.float32, device=pred.device)
    if ws is None:
        ws = loss_workspace(pred.device)
    L.check(L.load().a2f_voca_loss_fwd(pred.data_ptr(), gt.data_ptr(), rows, v3, k_rec, k_vel, out3.data_ptr(),
                                       ws.data_ptr(), ws.numel() * 8, _stream()), "a2f_voca_loss_fwd")
    return out3


def voca_loss_bwd(pred: torch.Tensor, gt: torch.Tensor, rows: int, v3: int, k_rec: float, k_vel: float,
                  gscale: Optional[torch.Tensor], dpred: torch.Tensor) -> torch.Tensor:
    _dev(pred, gt, dpred, gscale)
    L.check(L.load().a2f_voca_loss_bwd(pred.data_ptr(), gt.data_ptr(), rows, v3, k_rec, k_vel, L.ptr(gscale),
                                       dpred.data_ptr(), _stream()), "a2f_voca_loss_bwd")
    return dpred


def vertex_head_loss(z3: torch.Tensor, w3: torch.Tensor, bias: Optional[torch.Tensor], tmpl: Optional[torch.Tensor],
                     rows_per_tmpl: int, gt: torch.Tensor, dy: torch.Tensor, k_rec: float = 1.0, k_vel: float = 10.0,
                     pred: Optional[torch.Tensor] = None, ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Vertex head + VocaLoss in one pass (a2f_vertex_head_loss): z3 [rows,192] / w3 [V3,192] bf16x3 splits, gt [rows,V3] fp32,
    dy [rows, ld >= V3] bf16 receives d loss / d y (pad columns untouched).  -> out3 = (loss, rec, vel)."""
    _dev(z3, w3, bias, tmpl, gt, dy, pred, ws)
    rows, V3 = gt.shape
    if z3.dtype != torch.bfloat16 or w3.dtype != torch.bfloat16 or dy.dtype != torch.bfloat16 or gt.dtype != torch.float32:
        raise L.A2FError("vertex_head_loss: z3 / w3 / dy bf16, gt fp32")
    if not (z3.is_contiguous() and w3.is_contiguous() and gt.is_contiguous()) or dy.stride(1) != 1 or z3.shape[0] != rows \
            or w3.shape[0] != V3 or dy.shape[0] != rows or z3.shape[1] != w3.shape[1]:
        raise L.A2FError("vertex_head_loss: shape / layout mismatch")
    lib = L.load()
    if ws is None:
        ws = torch.empty((lib.a2f_vertex_head_loss_workspace_bytes() + 7) // 8, dtype=torch.float64, device=gt.device)
    out3 = torch.empty(3, dtype=torch.float32, device=gt.device)
    L.check(lib.a2f_vertex_head_loss(z3.data_ptr(), w3.data_ptr(), z3.shape[1], L.ptr(bias), L.ptr(tmpl), int(rows_per_tmpl),
                                     gt.data_ptr(), rows, V3, float(k_rec), float(k_vel), L.ptr(pred), dy.data_ptr(), dy.stride(0),
                                     out3.data_ptr(), ws.data_ptr(), ws.numel() * 8, _stream()), "a2f_vertex_head_loss")
    return out3


def split_bf16x3(x: torch.Tensor, is_weight: bool) -> torch.Tensor:
    """fp32 [rows,K] -> bf16 [rows,3K] error-compensated split (a2f_split_bf16x3)."""
    _dev(x)
    rows, K = x.shape
    out = torch.empty((rows, 3 * K), dtype=torch.bfloat16, device=x.device)
    L.check(L.load().a2f_split_bf16x3(x.data_ptr(), x.stride(0), out.data_ptr(), rows, K, 1 if is_weight else 0, _stream()),
            "a2f_split_bf16x3")
    return out


def pack_conv1d_weight(w: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    _dev(w)
    cout, cin, taps = w.shape
    out = torch.empty((cout, taps * cin), dtype=dtype, device=w.device)
    L.check(L.load().a2f_pack_conv1d_weight(w.contiguous().data_ptr(), out.data_ptr(), _dt(out), cout, cin, taps, _stream()),
            "a2f_pack_conv1d_weight")
    return out


def posconv_weight_shape(dtype: torch.dtype):
    """(kpad code, packed shape): fp32 SIMT layout [16][48 out][128 taps][48 in]; bf16 tcgen05 layout of posconv_tc.cu
    [16][128 taps][6 chunks][48 out][8 in] (kpad code 8)."""
    if dtype == torch.bfloat16:
        return 8, (16, 128, 6, 48, 8)
    return 48, (16, 48, 128, 48)


def pack_posconv_weight(g: torch.Tensor, v: torch.Tensor, dtype: torch.dtype, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _dev(g, v)
    kpad, shape = posconv_weight_shape(dtype)
    if out is None:
        out = torch.empty(shape, dtype=dtype, device=v.device)
    norm = torch.empty(128, dtype=torch.float32, device=v.device)
    L.check(L.load().a2f_pack_posconv_weight(g.contiguous().data_ptr(), v.contiguous().data_ptr(), out.data_ptr(), _dt(out),
                                             kpad, norm.data_ptr(), _stream()), "a2f_pack_posconv_weight")
    return out


def posconv(h: torch.Tensor, wp: torch.Tensor, bias: torch.Tensor, out: torch.Tensor, B: int, T: int, backend: int):
    _dev(h, wp, bias, out)
    prof = PROFILE is not None and backend == L.TCGEN05
    if prof:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
    L.check(L.load().a2f_posconv(h.data_ptr(), _dt(h), wp.data_ptr(), bias.data_ptr(), out.data_ptr(), _dt(out), B, T,
                                 backend, _stream()), "a2f_posconv")
    if prof:
        e.record()
        PROFILE.append(("gemm_tc", 2.0 * B * T * 768 * 48 * 128, s, e))
    return out


def audio_stats(audio: torch.Tensor) -> torch.Tensor:
    _dev(audio)
    B, N = audio.shape
    stats = torch.empty((B, 2), dtype=torch.float32, device=audio.device)
    L.check(L.load().a2f_audio_stats(audio.data_ptr(), B, N, stats.data_ptr(), _stream()), "a2f_audio_stats")
    return stats


def conv0_gn_gelu(audio: torch.Tensor, stats: torch.Tensor, w: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor,
                  dtype: torch.dtype) -> torch.Tensor:
    """-> channels-last [B, L0, 512]"""
    _dev(audio, stats, w, gamma, beta)
    B, N = audio.shape
    L0 = (N - 10) // 5 + 1
    lib = L.load()
    nbytes = lib.a2f_conv0_workspace_bytes(B, N)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=audio.device)
    out = torch.empty((B, L0, 512), dtype=dtype, device=audio.device)
    L.check(lib.a2f_conv0_gn_gelu(audio.data_ptr(), stats.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                  out.data_ptr(), _dt(out), B, N, ws.data_ptr(), ws.numel() * 8, _stream()),
            "a2f_conv0_gn_gelu")
    return out


def interp_ln(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, T: int, out_dtype: torch.dtype, eps: float = 1e-5):
    """[B,S,512] -> LayerNorm(linear_interpolation to T frames) [B,T,512]"""
    _dev(x, gamma, beta)
    B, S, Cc = x.shape
    out = torch.empty((B, T, Cc), dtype=out_dtype, device=x.device)
    L.check(L.load().a2f_interp_ln(x.data_ptr(), _dt(x), gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr(), _dt(out),
                                   B, S, T, Cc, _stream()), "a2f_interp_ln")
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, out: torch.Tensor, eps: float = 1e-5,
              out2: Optional[torch.Tensor] = None) -> torch.Tensor:
    _dev(x, gamma, beta, out, out2)
    rows, Cc = x.shape
    L.check(L.load().a2f_layernorm(x.data_ptr(), _dt(x), gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr(), _dt(out),
                                   L.ptr(out2), _dt(out2) if out2 is not None else 0, rows, Cc, _stream()), "a2f_layernorm")
    return out


def mha(qkv: torch.Tensor, out: torch.Tensor, B: int, T: int, H: int = 12, D: int = 64, scale: float = 0.125):
    _dev(qkv, out)
    L.check(L.load().a2f_mha_fwd(qkv.data_ptr(), out.data_ptr(), _dt(qkv), B, T, H, D, scale, _stream()), "a2f_mha_fwd")
    return out


def a2m_assemble(x: torch.Tensor, one_hot: torch.Tensor) -> torch.Tensor:
    """x [B,52,32], one_hot [B,n] -> zero-left-padded single-channel input [B,64,33] (a2f_a2m_assemble)."""
    _dev(x, one_hot)
    B = x.shape[0]
    out = torch.empty((B, 64, 33), dtype=torch.float32, device=x.device)
    L.check(L.load().a2f_a2m_assemble(x.data_ptr(), one_hot.data_ptr(), one_hot.shape[1], out.data_ptr(), B, _stream()),
            "a2f_a2m_assemble")
    return out


def channel_affine(buf: torch.Tensor, offset: int, scale: torch.Tensor, shift: torch.Tensor, C_: int, rows_per_batch: int,
                   ld: int, batch_stride: int, batches: int) -> None:
    _dev(buf, scale, shift)
    L.check(L.load().a2f_channel_affine(buf.data_ptr() + offset * buf.element_size(), _dt(buf), scale.data_ptr(),
                                        shift.data_ptr(), C_, rows_per_batch, ld, batch_stride, batches, _stream()),
            "a2f_channel_affine")


def im2col1d_split(x: torch.Tensor, outer: int, outer_stride: int, ld: int, C_: int, L_: int, taps: int, stride: int, pad: int,
                   kpad: int, scale: Optional[torch.Tensor] = None, shift: Optional[torch.Tensor] = None,
                   x_offset: int = 0) -> torch.Tensor:
    """fp32 channels-last [outer, L, C] -> bf16 [outer*L_out, 3*kpad] im2col rows in the hi|lo|hi split (a2f_im2col1d_split)."""
    _dev(x, scale, shift)
    L_out = (L_ + 2 * pad - taps) // stride + 1
    out = torch.empty((outer * L_out, 3 * kpad), dtype=torch.bfloat16, device=x.device)
    L.check(L.load().a2f_im2col1d_split(x.data_ptr() + x_offset * 4, outer, outer_stride, ld, C_, L_, taps, stride, pad,
                                        L.ptr(scale), L.ptr(shift), kpad, out.data_ptr(), _stream()), "a2f_im2col1d_split")
    return out


def im2col1d(x: torch.Tensor, outer: int, outer_stride: int, ld: int, C_: int, L_: int, taps: int, stride: int, pad: int,
             kpad: int, split: bool, scale: Optional[torch.Tensor] = None, shift: Optional[torch.Tensor] = None,
             x_offset: int = 0) -> torch.Tensor:
    """im2col rows of a 1-D conv over channels-last fp32 [outer, L, C]: bf16 hi|lo|hi split (tcgen05 path) or plain fp32."""
    if split:
        return im2col1d_split(x, outer, outer_stride, ld, C_, L_, taps, stride, pad, kpad, scale, shift, x_offset)
    _dev(x, scale, shift)
    L_out = (L_ + 2 * pad - taps) // stride + 1
    out = torch.empty((outer * L_out, kpad), dtype=torch.float32, device=x.device)
    L.check(L.load().a2f_im2col1d(x.data_ptr() + x_offset * 4, outer, outer_stride, ld, C_, L_, taps, stride, pad, L.ptr(scale),
                                  L.ptr(shift), kpad, out.data_ptr(), _stream()), "a2f_im2col1d")
    return out


def col2im1d(dcol: torch.Tensor, dx: torch.Tensor, outer: int, outer_stride: int, ld: int, C_: int, L_: int, taps: int, stride: int,
             pad: int, x_offset: int = 0) -> torch.Tensor:
    """adjoint of im2col1d(split=False): writes every valid element (l < L, c < C) of dx, laid out like im2col1d's x"""
    _dev(dcol, dx)
    L_out = (L_ + 2 * pad - taps) // stride + 1
    if dcol.dim() != 2 or dcol.shape[0] != outer * L_out or dcol.stride(0) != dcol.shape[1] or \
            dx.numel() < x_offset + (outer - 1) * outer_stride + (L_ - 1) * ld + C_:
        raise L.A2FError("col2im1d: dcol must be a dense [outer*L_out, kpad] matrix and dx must hold the strided layout")
    L.check(L.load().a2f_col2im1d(dx.data_ptr() + x_offset * 4, outer, outer_stride, ld, C_, L_, taps, stride, pad, None, None,
                                  dcol.shape[1], dcol.data_ptr(), _stream()), "a2f_col2im1d")
    return dx


def transpose_batched(x: torch.Tensor) -> torch.Tensor:
    """[B, R, C] fp32 -> [B, C, R]"""
    _dev(x)
    B, R, C_ = x.shape
    y = torch.empty((B, C_, R), dtype=torch.float32, device=x.device)
    L.check(L.load().a2f_transpose_batched(x.data_ptr(), y.data_ptr(), B, R, C_, _stream()), "a2f_transpose_batched")
    return y


def lstm_recurrence(xp: torch.Tensor, whh_t: torch.Tensor, B: int, T: int, hidden: int,
                    whh: Optional[torch.Tensor] = None) -> torch.Tensor:
    """xp [B,T,4H] input projections (+ both biases), whh_t = W_hh^T [H,4H], whh = W_hh [4H,H] (cluster kernel) -> h [B,T,H]"""
    _dev(xp, whh_t, whh)
    if whh is None:
        whh = whh_t.t().contiguous()
    h = torch.empty((B, T, hidden), dtype=torch.float32, device=xp.device)
    L.check(L.load().a2f_lstm_recurrence(xp.data_ptr(), whh_t.data_ptr(), whh.data_ptr(), h.data_ptr(), B, T, hidden, _stream()),
            "a2f_lstm_recurrence")
    return h


def song2face_resize(h: torch.Tensor, out_h: int) -> torch.Tensor:
    _dev(h)
    B, T, hid = h.shape
    out = torch.empty((B, out_h, T), dtype=torch.float32, device=h.device)
    L.check(L.load().a2f_song2face_resize(h.data_ptr(), B, T, hid, out_h, out.data_ptr(), _stream()), "a2f_song2face_resize")
    return out


def song2face_resize_bwd(dout: torch.Tensor, hidden: int) -> torch.Tensor:
    """adjoint of song2face_resize: dout [B, out_h, T] -> dh [B, T, hidden]"""
    _dev(dout)
    B, out_h, T = dout.shape
    dh = torch.empty((B, T, hidden), dtype=torch.float32, device=dout.device)
    L.check(L.load().a2f_song2face_resize_bwd(dout.data_ptr(), B, T, hidden, out_h, dh.data_ptr(), _stream()),
            "a2f_song2face_resize_bwd")
    return dh


def lstm_recurrence_train(xp: torch.Tensor, whh: torch.Tensor, B: int, T: int, hidden: int):
    """training forward of the recurrence: xp [B,T,4H], whh = W_hh [4H,H] -> (h [B,T,H], gates [B,T,4H], c [B,T,H])"""
    _dev(xp, whh)
    h = torch.empty((B, T, hidden), dtype=torch.float32, device=xp.device)
    gates = torch.empty((B, T, 4 * hidden), dtype=torch.float32, device=xp.device)
    cell = torch.empty((B, T, hidden), dtype=torch.float32, device=xp.device)
    L.check(L.load().a2f_lstm_recurrence_train(xp.data_ptr(), whh.data_ptr(), h.data_ptr(), gates.data_ptr(), cell.data_ptr(), B, T,
                                               hidden, _stream()), "a2f_lstm_recurrence_train")
    return h, gates, cell


def lstm_bptt(dh_out: torch.Tensor, gates: torch.Tensor, cell: torch.Tensor, whh: torch.Tensor) -> torch.Tensor:
    """dh_out [B,T,H], the saved gates / c, W_hh [4H,H] -> dgates [B,T,4H] (gradient of the pre-activation gates)"""
    _dev(dh_out, gates, cell, whh)
    B, T, hidden = cell.shape
    for t, shape in ((dh_out, (B, T, hidden)), (gates, (B, T, 4 * hidden)), (whh, (4 * hidden, hidden))):
        if tuple(t.shape) != shape or not t.is_contiguous():
            raise L.A2FError(f"lstm_bptt: expected a contiguous tensor of shape {shape}, got {tuple(t.shape)}")
    dgates = torch.empty((B, T, 4 * hidden), dtype=torch.float32, device=cell.device)
    L.check(L.load().a2f_lstm_bptt(dh_out.data_ptr(), gates.data_ptr(), cell.data_ptr(), whh.data_ptr(), dgates.data_ptr(), B, T,
                                   hidden, _stream()), "a2f_lstm_bptt")
    return dgates


def a2m_mlp(feat: torch.Tensor, extra: torch.Tensor, fc0, fc1, fc2, ldz: int = 64) -> torch.Tensor:
    """z = fc2(tanh(fc1(fc0(cat(feat, extra))))) zero-padded to ldz columns (a2f_a2m_mlp); fc* are nn.Linear modules."""
    _dev(feat, extra)
    B = feat.shape[0]
    z = torch.empty((B, ldz), dtype=torch.float32, device=feat.device)
    w = [t.detach().contiguous() for fc in (fc0, fc1, fc2) for t in (fc.weight, fc.bias)]
    L.check(L.load().a2f_a2m_mlp(feat.data_ptr(), feat.stride(0), feat.shape[1], extra.data_ptr(), extra.shape[1],
                                 w[0].data_ptr(), w[1].data_ptr(), w[0].shape[0], w[2].data_ptr(), w[3].data_ptr(), w[2].shape[0],
                                 w[4].data_ptr(), w[5].data_ptr(), w[4].shape[0], z.data_ptr(), ldz, B, _stream()), "a2f_a2m_mlp")
    return z


def pack_feedback(vm_w, vm_b, vmr_w, vmr_b, out=None):
    _dev(vm_w, vm_b, vmr_w, vmr_b)
    if out is None:
        wc = torch.empty((64, 64), dtype=torch.float32, device=vm_w.device)
        bc = torch.empty((64,), dtype=torch.float32, device=vm_w.device)
    else:
        wc, bc = out
    L.check(L.load().a2f_pack_feedback(vm_w.data_ptr(), vm_b.data_ptr(), vmr_w.data_ptr(), vmr_b.data_ptr(),
                                       vmr_w.shape[0], wc.data_ptr(), bc.data_ptr(), _stream()), "a2f_pack_feedback")
    return wc, bc


def pack_decoder_fold(sa_in_w: torch.Tensor, wc: torch.Tensor, pe: torch.Tensor, period: int, fold_w: torch.Tensor,
                      fold_pe: torch.Tensor) -> None:
    """fold_w [192,64] = in_proj @ Wc, fold_pe [period,192] = pe @ in_proj^T (a2f_pack_decoder_fold; run after pack_feedback)."""
    _dev(sa_in_w, wc, pe, fold_w, fold_pe)
    if tuple(fold_w.shape) != (192, 64) or tuple(fold_pe.shape) != (period, 192) or pe.reshape(-1).numel() < period * 64:
        raise L.A2FError("pack_decoder_fold: shape mismatch")
    L.check(L.load().a2f_pack_decoder_fold(sa_in_w.data_ptr(), wc.data_ptr(), pe.data_ptr(), int(period), fold_w.data_ptr(),
                                           fold_pe.data_ptr(), _stream()), "a2f_pack_decoder_fold")


def pack_cross_attention(in_proj_w, in_proj_b, out_w, out_b, afm_w, afm_b, W: torch.Tensor, b: torch.Tensor) -> None:
    """W[64,Kin], b[64] = out_proj(v_proj(audio_feature_map(.))) folded in fp64 (a2f_pack_cross_attention).  in_proj_*: the
    packed [192,64] / [192] multihead_attn.in_proj parameters (rows 128..191 = v)."""
    _dev(in_proj_w, in_proj_b, out_w, out_b, afm_w, afm_b, W, b)
    for t in (in_proj_w, in_proj_b, out_w, out_b, afm_w, afm_b):
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise L.A2FError("pack_cross_attention takes contiguous fp32 parameters")
    L.check(L.load().a2f_pack_cross_attention(in_proj_w.data_ptr() + 128 * 64 * 4, in_proj_b.data_ptr() + 128 * 4, out_w.data_ptr(),
                                              out_b.data_ptr(), afm_w.data_ptr(), afm_b.data_ptr(), afm_w.shape[1], W.data_ptr(),
                                              _dt(W), b.data_ptr(), _stream()), "a2f_pack_cross_attention")


def decoder_rollout(wstruct: "L.DecoderWeights", memory: torch.Tensor, one_hot: torch.Tensor, period: int, B: int, T: int,
                    memory_is_ca: bool = False):
    """memory [B,T,64] fp32 -> decoder states D [B,T,64] fp32 (a2f_decoder_rollout); memory_is_ca: `memory` already holds
    the cross-attention vectors out_proj(v_proj(audio_feature_map(h))) (a2f_decoder_rollout_ca)."""
    _dev(memory, one_hot)
    lib = L.load()
    nbytes = lib.a2f_decoder_workspace_bytes(B, T)
    ws = torch.empty((nbytes + 15) // 16 * 4, dtype=torch.float32, device=memory.device)
    D = torch.empty((B, T, 64), dtype=torch.float32, device=memory.device)
    fn = lib.a2f_decoder_rollout_ca if memory_is_ca else lib.a2f_decoder_rollout
    L.check(fn(C.byref(wstruct), memory.data_ptr(), one_hot.data_ptr(), one_hot.shape[1], period,
               D.data_ptr(), B, T, ws.data_ptr(), ws.numel() * 4, _stream()), "a2f_decoder_rollout")
    return D


def head_stream_supported(B: int, T: int, v3: int) -> bool:
    """When the streamed vertex head (rollout_and_head_stream) pays: 32 or 64 utterances (the head gets the SMs the rollout
    leaves idle: with 128 utterances that would be 20 of 148) and clips below 900 frames (from there on the rollout spreads an
    utterance over a CTA cluster, which the streaming kernel does not do); the kernel itself needs T * V3 < 2^25."""
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return B in (32, 64) and T < 900 and L.load().a2f_vertex_head_stream_rows(int(B), int(T)) > 0 and \
        T * v3 < (1 << 25) and 2 * B <= sms


class _StreamPair:
    """The side stream (per device) on which the vertex head follows the rollout."""
    _side = {}

    @classmethod
    def side(cls, device) -> "torch.cuda.Stream":
        key = torch.device(device).index
        if key not in cls._side:
            cls._side[key] = torch.cuda.Stream(device=device)
        return cls._side[key]


def rollout_and_head_stream(wstruct: "L.DecoderWeights", ca: torch.Tensor, one_hot: torch.Tensor, period: int, B: int, T: int,
                            w3: torch.Tensor, bias: torch.Tensor, tmpl: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """Decoder rollout and vertex head as two kernels that run AT THE SAME TIME (a2f_decoder_rollout_stream on the current
    stream, a2f_vertex_head_stream on a side stream): the rollout keeps one SM per utterance busy for T dependent steps, the
    head follows it frame group by frame group on the other SMs, so only the last group's tiles remain when the rollout
    ends.  ca [B*T,64] fp32 cross-attention vectors, w3 [V3,192] bf16 (hi|hi|lo), tmpl [B,V3] fp32, out [B*T,V3] fp32 dense.
    Returns D [B,T,64].  Works inside CUDA-graph capture (the side stream forks from and joins the capturing stream)."""
    _dev(ca, one_hot, w3, bias, tmpl, out)
    lib = L.load()
    v3 = w3.shape[0]
    rows = lib.a2f_vertex_head_stream_rows(B, T)
    if rows <= 0 or out.stride(0) != v3 or not out.is_contiguous() or tuple(tmpl.shape) != (B, v3) or w3.shape[1] != 192:
        raise L.A2FError("rollout_and_head_stream: unsupported shapes")
    dev = ca.device
    nbytes = lib.a2f_decoder_workspace_bytes(B, T)
    ws = torch.empty((nbytes + 15) // 16 * 4, dtype=torch.float32, device=dev)
    D = torch.empty((B, T, 64), dtype=torch.float32, device=dev)
    z3 = torch.empty((rows, 192), dtype=torch.bfloat16, device=dev)     # (rows past T*B feed accumulator rows nobody stores)
    done = torch.zeros(T, dtype=torch.int32, device=dev)
    cur = torch.cuda.current_stream(dev)
    side = _StreamPair.side(dev)
    side.wait_stream(cur)                                   # fork: operands, zeroed counters
    L.check(lib.a2f_decoder_rollout_stream(C.byref(wstruct), ca.data_ptr(), one_hot.data_ptr(), one_hot.shape[1], period,
                                           D.data_ptr(), B, T, ws.data_ptr(), ws.numel() * 4, z3.data_ptr(), done.data_ptr(),
                                           cur.cuda_stream), "a2f_decoder_rollout_stream")
    with torch.cuda.stream(side):
        L.check(lib.a2f_vertex_head_stream(z3.data_ptr(), w3.data_ptr(), 192, L.ptr(bias), tmpl.data_ptr(), B, T, v3,
                                           out.data_ptr(), done.data_ptr(), B, side.cuda_stream), "a2f_vertex_head_stream")
    cur.wait_stream(side)                                   # join (every tensor used on the side stream is released after it)
    return D


# ---------------------------------------------------------------------------------------------------------------
# training step (backward-pass kernels, csrc/train.cu / attention.cu / decoder_bwd.cu)
# ---------------------------------------------------------------------------------------------------------------
def act_fwd(z: torch.Tensor, act: int, out_dtype: Optional[torch.dtype] = None, resid: Optional[torch.Tensor] = None,
            out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _dev(z, resid, out)
    if out is None:
        out = torch.empty(z.shape, dtype=out_dtype or z.dtype, device=z.device)
    if resid is not None and resid.dtype != out.dtype:
        raise L.A2FError("act_fwd: resid must have the output dtype")
    L.check(L.load().a2f_act_fwd(z.data_ptr(), _dt(z), L.ptr(resid), out.data_ptr(), _dt(out), z.numel(), act, _stream()),
            "a2f_act_fwd")
    return out


def act_bwd(dy: torch.Tensor, z: torch.Tensor, act: int, out_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    _dev(dy, z)
    out = torch.empty(z.shape, dtype=out_dtype or z.dtype, device=z.device)
    L.check(L.load().a2f_act_bwd(dy.data_ptr(), _dt(dy), z.data_ptr(), _dt(z), out.data_ptr(), _dt(out), z.numel(), act,
                                 _stream()), "a2f_act_bwd")
    return out


def cast_rows(x: torch.Tensor, out_dtype: torch.dtype, ld_out: int) -> torch.Tensor:
    """[rows, cols] -> [rows, ld_out] converted, zero padded on the right."""
    _dev(x)
    rows, cols = x.shape
    out = torch.empty((rows, ld_out), dtype=out_dtype, device=x.device)
    L.check(L.load().a2f_cast_rows(x.data_ptr(), _dt(x), x.stride(0), out.data_ptr(), _dt(out), ld_out, rows, cols, _stream()),
            "a2f_cast_rows")
    return out


def transpose_cast(w: torch.Tensor, out_dtype: torch.dtype, R: Optional[int] = None, Cc: Optional[int] = None,
                   ld_r: Optional[int] = None, ld_c: int = 1, offset: int = 0, out: Optional[torch.Tensor] = None,
                   ldo: Optional[int] = None, out_offset: int = 0) -> torch.Tensor:
    """out[c, r] = w.flat[offset + r*ld_r + c*ld_c]  (fp32 in, fp32/bf16 out)."""
    _dev(w)
    if w.dtype != torch.float32:
        raise L.A2FError("transpose_cast takes fp32 input")
    R = int(R if R is not None else w.shape[0])
    Cc = int(Cc if Cc is not None else w.shape[1])
    ld_r = int(ld_r if ld_r is not None else w.stride(0))
    if out is None:
        out = torch.empty((Cc, R), dtype=out_dtype, device=w.device)
    ldo = int(ldo if ldo is not None else out.stride(0))
    L.check(L.load().a2f_transpose_cast(w.data_ptr() + 4 * offset, ld_r, ld_c, R, Cc,
                                        out.data_ptr() + out_offset * out.element_size(), _dt(out), ldo, _stream()),
            "a2f_transpose_cast")
    return out


class PackPlan:
    """A recorded list of strided fp32 -> fp32/bf16 copies executed by ONE kernel launch (a2f_strided_copy_jobs).

    The drop-in modules derive every packed GEMM operand (bf16 casts, W^T data-gradient operands, implicit-GEMM conv
    layouts, the fused QKV weight) from the fp32 master parameters.  Source and destination pointers are stable across
    optimizer steps (parameters are updated in place, destinations are owned by the plan's user), so the job table is
    uploaded once and `run()` re-derives all operands after every step."""

    def __init__(self, device):
        self.device = device
        self.jobs = []
        self.keep = []          # tensors the jobs point into (kept alive with the plan)
        self.table = None
        self.total_tiles = 0

    def add(self, src: torch.Tensor, dst: torch.Tensor, R: int, Cc: int, ld_r: int, ld_c: int, ldo_r: int, ldo_c: int,
            src_off: int = 0, dst_off: int = 0) -> None:
        """dst.flat[dst_off + r*ldo_r + c*ldo_c] = src.flat[src_off + r*ld_r + c*ld_c], r < R, c < Cc."""
        _dev(src, dst)
        if src.dtype != torch.float32 or dst.dtype not in (torch.float32, torch.bfloat16):
            raise L.A2FError("PackPlan copies fp32 sources into fp32 / bf16 destinations")
        if self.table is not None:
            raise L.A2FError("PackPlan is already finalised")
        j = L.CopyJob()
        j.src = src.data_ptr() + 4 * src_off
        j.dst = dst.data_ptr() + dst.element_size() * dst_off
        j.ld_r, j.ld_c, j.ldo_r, j.ldo_c = int(ld_r), int(ld_c), int(ldo_r), int(ldo_c)
        j.R, j.C, j.dst_dtype = int(R), int(Cc), _dt(dst)
        j.tile0 = self.total_tiles
        self.total_tiles += ((int(R) + 31) // 32) * ((int(Cc) + 31) // 32)
        self.jobs.append(j)
        self.keep += [src, dst]

    def cast(self, src: torch.Tensor, dst: torch.Tensor, dst_off: int = 0) -> None:
        """dst.flat[dst_off:dst_off + src.numel()] = src (row-major, contiguous)."""
        cols = src.shape[-1]
        rows = src.numel() // cols
        self.add(src, dst, rows, cols, cols, 1, cols, 1, dst_off=dst_off)

    def transpose(self, src: torch.Tensor, dst: torch.Tensor, ldo: Optional[int] = None, dst_off: int = 0, R=None, Cc=None,
                  ld_r=None, ld_c: int = 1, src_off: int = 0) -> None:
        """dst[c, r] = src.flat[src_off + r*ld_r + c*ld_c]   (same contract as transpose_cast)."""
        R = int(R if R is not None else src.shape[0])
        Cc = int(Cc if Cc is not None else src.shape[1])
        ld_r = int(ld_r if ld_r is not None else src.stride(0))
        ldo = int(ldo if ldo is not None else dst.stride(0))
        self.add(src, dst, R, Cc, ld_r, ld_c, 1, ldo, src_off=src_off, dst_off=dst_off)

    def finalize(self) -> "PackPlan":
        if not self.jobs:
            raise L.A2FError("empty PackPlan")
        arr = (L.CopyJob * len(self.jobs))(*self.jobs)
        raw = bytes(arr)
        host = torch.frombuffer(bytearray(raw), dtype=torch.uint8)
        self.table = host.to(self.device)
        return self

    def run(self) -> None:
        if self.table is None:
            self.finalize()
        L.check(L.load().a2f_strided_copy_jobs(self.table.data_ptr(), len(self.jobs), self.total_tiles, _stream()),
                "a2f_strided_copy_jobs")


def colsum(x: torch.Tensor, out: torch.Tensor, rows: Optional[int] = None, cols: Optional[int] = None,
           ld: Optional[int] = None) -> torch.Tensor:
    """out[n] += sum_m x[m, n]"""
    _dev(x, out)
    rows = int(rows if rows is not None else x.shape[0])
    cols = int(cols if cols is not None else x.shape[1])
    L.check(L.load().a2f_colsum(x.data_ptr(), _dt(x), int(ld if ld is not None else x.stride(0)), rows, cols, out.data_ptr(),
                                _stream()), "a2f_colsum")
    return out


def colsum3(x: torch.Tensor, outs) -> None:
    """outs[i][n] += sum_m x[m, i*seg + n] for the three column segments of a fused [M, 3*seg] gradient, one launch."""
    _dev(x, *outs)
    seg = x.shape[1] // 3
    L.check(L.load().a2f_colsum3(x.data_ptr(), _dt(x), x.stride(0), x.shape[0], seg, outs[0].data_ptr(), outs[1].data_ptr(),
                                 outs[2].data_ptr(), _stream()), "a2f_colsum3")


def _dropout_args(p: float, site: int, seed_offset: Optional[torch.Tensor]) -> "L.DropoutArgs":
    if seed_offset is not None:
        _dev(seed_offset)
        if seed_offset.dtype != torch.int64 or seed_offset.numel() != 2 or not seed_offset.is_contiguous():
            raise L.A2FError("dropout: seed_offset is a contiguous int64 device tensor {seed, offset}")
    return L.DropoutArgs(float(p), int(site), L.ptr(seed_offset))


def dropout_mask(p: float, site: int, seed_offset: torch.Tensor, shape) -> torch.Tensor:
    """Keep mask (uint8, 1 = kept) of one dropout site over its logical tensor `shape` (RNG contract, include/a2f.h)."""
    mask = torch.empty(tuple(shape), dtype=torch.uint8, device=seed_offset.device)
    L.check(L.load().a2f_dropout_mask(C.byref(_dropout_args(p, site, seed_offset)), mask.numel(), mask.data_ptr(),
                                      _stream()), "a2f_dropout_mask")
    return mask


def dropout_apply(x: torch.Tensor, p: float, site: int, seed_offset: torch.Tensor, resid: Optional[torch.Tensor] = None,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = drop(x) [+ resid] (out may be x or resid); also the backward of the site when x is its gradient."""
    _dev(x, resid, out)
    if out is None:
        out = torch.empty_like(x)
    for t in (x, resid, out):
        if t is not None and (t.dtype != x.dtype or not t.is_contiguous() or t.numel() != x.numel()):
            raise L.A2FError("dropout_apply: x, resid and out are contiguous tensors of one dtype and size")
    L.check(L.load().a2f_dropout_apply(x.data_ptr(), L.ptr(resid), out.data_ptr(), _dt(x), x.numel(),
                                       C.byref(_dropout_args(p, site, seed_offset)), _stream()), "a2f_dropout_apply")
    return out


def spec_mask_fwd(h: torch.Tensor, mask_u8: torch.Tensor, embed: torch.Tensor) -> torch.Tensor:
    """h[mask] = embed, in place (ref:src/model/wav2vec.py:159-161).  h [rows, cols], mask_u8 uint8 [rows]."""
    _dev(h, mask_u8, embed)
    rows, cols = h.shape
    L.check(L.load().a2f_spec_mask_fwd(h.data_ptr(), _dt(h), mask_u8.data_ptr(), embed.data_ptr(), rows, cols, _stream()),
            "a2f_spec_mask_fwd")
    return h


def spec_mask_bwd(dh: torch.Tensor, mask_u8: torch.Tensor, dembed: torch.Tensor) -> torch.Tensor:
    """dembed += sum of the masked rows of dh; those rows of dh are zeroed in place."""
    _dev(dh, mask_u8, dembed)
    rows, cols = dh.shape
    L.check(L.load().a2f_spec_mask_bwd(dh.data_ptr(), _dt(dh), mask_u8.data_ptr(), dembed.data_ptr(), rows, cols, _stream()),
            "a2f_spec_mask_bwd")
    return dh


def layernorm_bwd(dy: torch.Tensor, x: torch.Tensor, gamma: torch.Tensor, dgamma: torch.Tensor, dbeta: torch.Tensor,
                  dbias: Optional[torch.Tensor] = None, eps: float = 1e-5) -> torch.Tensor:
    _dev(dy, x, gamma, dgamma, dbeta, dbias)
    rows, Cc = x.shape
    dx = torch.empty_like(x)
    L.check(L.load().a2f_layernorm_bwd(dy.data_ptr(), _dt(dy), x.data_ptr(), _dt(x), gamma.data_ptr(), eps, dx.data_ptr(),
                                       _dt(dx), dgamma.data_ptr(), dbeta.data_ptr(), L.ptr(dbias), rows, Cc, _stream()),
            "a2f_layernorm_bwd")
    return dx


def interp_ln_bwd(x: torch.Tensor, dy: torch.Tensor, gamma: torch.Tensor, dgamma: torch.Tensor, dbeta: torch.Tensor,
                  eps: float = 1e-5) -> torch.Tensor:
    """x [B,S,512] saved input, dy [B,T,512] -> fp32 gradient wrt x."""
    _dev(x, dy, gamma, dgamma, dbeta)
    B, S, Cc = x.shape
    T = dy.shape[1]
    din = torch.zeros((B, S, Cc), dtype=torch.float32, device=x.device)
    L.check(L.load().a2f_interp_ln_bwd(x.data_ptr(), _dt(x), dy.data_ptr(), _dt(dy), gamma.data_ptr(), eps, din.data_ptr(),
                                       dgamma.data_ptr(), dbeta.data_ptr(), B, S, T, Cc, _stream()), "a2f_interp_ln_bwd")
    return din


def padded_rows(B: int, rows: int, C_: int, dtype: torch.dtype, device) -> torch.Tensor:
    """[B, rows, C] activation followed by one zeroed spare row.  The weight-gradient GEMM of a stride-2 Conv1d reads
    its input as rows of 2*C elements (a2f_gemm_wgrad, x_row_stride = 2*C): when `rows` is odd the last such row of
    the LAST utterance extends C elements past the tensor; they are multiplied by zero-filled dY rows, so they must be
    finite (0 * NaN = NaN inside the MMA)."""
    flat = torch.empty(B * rows * C_ + C_, dtype=dtype, device=device)
    flat[B * rows * C_:].zero_()
    return flat[: B * rows * C_].view(B, rows, C_)


def conv0_gn_gelu_auto(audio: torch.Tensor, w: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, dtype: torch.dtype):
    """Processor normalisation + conv0 + GroupNorm + GELU from one pass over the raw audio (a2f_conv0_gn_gelu_auto).
    -> (channels-last [B, L0, 512], stats [B,2])"""
    _dev(audio, w, gamma, beta)
    B, N = audio.shape
    L0 = (N - 10) // 5 + 1
    lib = L.load()
    nbytes = lib.a2f_conv0_auto_workspace_bytes(B, N)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=audio.device)
    stats = torch.empty((B, 2), dtype=torch.float32, device=audio.device)
    out = torch.empty((B, L0, 512), dtype=dtype, device=audio.device)
    L.check(lib.a2f_conv0_gn_gelu_auto(audio.data_ptr(), stats.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                       out.data_ptr(), _dt(out), B, N, ws.data_ptr(), ws.numel() * 8, _stream()),
            "a2f_conv0_gn_gelu_auto")
    return out, stats


def conv0_gn_gelu_train(audio, stats, w, gamma, beta, dtype):
    """conv0_gn_gelu that also returns the workspace (it holds the GroupNorm statistics the backward needs)."""
    _dev(audio, stats, w, gamma, beta)
    B, N = audio.shape
    L0 = (N - 10) // 5 + 1
    lib = L.load()
    nbytes = lib.a2f_conv0_workspace_bytes(B, N)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=audio.device)
    out = padded_rows(B, L0, 512, dtype, audio.device)
    L.check(lib.a2f_conv0_gn_gelu(audio.data_ptr(), stats.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                  out.data_ptr(), _dt(out), B, N, ws.data_ptr(), ws.numel() * 8, _stream()),
            "a2f_conv0_gn_gelu")
    return out, ws


def conv0_bwd(audio, stats, w, gamma, beta, ws, da, dw, dgamma, dbeta):
    _dev(audio, stats, w, gamma, beta, ws, da, dw, dgamma, dbeta)
    B, N = audio.shape
    lib = L.load()
    off = lib.a2f_conv0_gn_offset(B, N)
    nb = lib.a2f_conv0_bwd_workspace_bytes(B)
    scratch = torch.empty((nb + 3) // 4, dtype=torch.float32, device=audio.device)
    L.check(lib.a2f_conv0_bwd(audio.data_ptr(), stats.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                              ws.data_ptr() + off, da.data_ptr(), _dt(da), B, N, dw.data_ptr(), dgamma.data_ptr(),
                              dbeta.data_ptr(), scratch.data_ptr(), scratch.numel() * 4, _stream()), "a2f_conv0_bwd")


def pack_posconv_weights_train(g: torch.Tensor, v: torch.Tensor, dtype: torch.dtype, out=None):
    """-> (forward packed weight, data-gradient packed weight)"""
    _dev(g, v)
    kpad, shape = posconv_weight_shape(dtype)
    lib = L.load()
    if out is None:
        fwd = torch.empty(shape, dtype=dtype, device=v.device)
        bwd = torch.empty(shape, dtype=dtype, device=v.device)
    else:
        fwd, bwd = out
    norm = torch.empty(128, dtype=torch.float32, device=v.device)
    gc, vc = g.contiguous(), v.contiguous()
    L.check(lib.a2f_pack_posconv_weight(gc.data_ptr(), vc.data_ptr(), fwd.data_ptr(), _dt(fwd), kpad, norm.data_ptr(), _stream()),
            "a2f_pack_posconv_weight")
    L.check(lib.a2f_pack_posconv_dgrad_weight(gc.data_ptr(), vc.data_ptr(), bwd.data_ptr(), _dt(bwd), kpad, norm.data_ptr(),
                                              _stream()), "a2f_pack_posconv_dgrad_weight")
    return fwd, bwd


def posconv_pre(h, wp, bias, B, T, backend):
    _dev(h, wp, bias)
    pc = torch.empty_like(h)
    L.check(L.load().a2f_posconv_pre(h.data_ptr(), _dt(h), wp.data_ptr(), bias.data_ptr(), pc.data_ptr(), B, T, backend,
                                     _stream()), "a2f_posconv_pre")
    return pc


def posconv_dgrad(dpc, wd, dout, B, T, backend):
    _dev(dpc, wd, dout)
    dh = torch.empty_like(dpc)
    L.check(L.load().a2f_posconv_dgrad(dpc.data_ptr(), _dt(dpc), wd.data_ptr(), L.ptr(dout), dh.data_ptr(), B, T, backend,
                                       _stream()), "a2f_posconv_dgrad")
    return dh


def posconv_wgrad(dpc, h, B, T, backend):
    """-> fp32 gradient wrt the effective conv weight in the packed layout [16][48][128][48]"""
    _dev(dpc, h)
    dwp = torch.zeros((16, 48, 128, 48), dtype=torch.float32, device=h.device)
    L.check(L.load().a2f_posconv_wgrad(dpc.data_ptr(), h.data_ptr(), _dt(h), dwp.data_ptr(), B, T, backend, _stream()),
            "a2f_posconv_wgrad")
    return dwp


def weight_norm_bwd(dwp, v, g, dv, dg):
    _dev(dwp, v, g, dv, dg)
    ws = torch.empty(256, dtype=torch.float64, device=v.device)
    L.check(L.load().a2f_weight_norm_bwd(dwp.data_ptr(), v.data_ptr(), g.data_ptr(), dv.data_ptr(), dg.data_ptr(),
                                         ws.data_ptr(), 256 * 8, _stream()), "a2f_weight_norm_bwd")


def mha_lse(qkv, out, lse, B, T, H=12, D=64, scale=0.125, out_f32: Optional[torch.Tensor] = None, dropout=None):
    """training forward: also the row log-sum-exp and (bf16 path, optional) the un-rounded fp32 output.
    dropout: None, or (p, site, seed_offset) -- attention-probability dropout (a2f_mha_fwd_train_dropout)."""
    _dev(qkv, out, lse, out_f32)
    if out_f32 is not None and (out_f32.dtype != torch.float32 or qkv.dtype != torch.bfloat16):
        raise L.A2FError("out_f32 is the fp32 side output of the bf16 attention kernel")
    if dropout is None:
        L.check(L.load().a2f_mha_fwd_train(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), L.ptr(out_f32), _dt(qkv), B, T, H,
                                           D, scale, _stream()), "a2f_mha_fwd_train")
        return out
    L.check(L.load().a2f_mha_fwd_train_dropout(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), L.ptr(out_f32), _dt(qkv), B, T,
                                               H, D, scale, C.byref(_dropout_args(*dropout)), _stream()),
            "a2f_mha_fwd_train_dropout")
    return out


def mha_bwd(qkv, out, dout, lse, B, T, H=12, D=64, scale=0.125, out_f32: Optional[torch.Tensor] = None, dropout=None):
    """dropout: the forward's (p, site, seed_offset), whose mask the backward regenerates."""
    _dev(qkv, out, dout, lse, out_f32)
    dqkv = torch.empty_like(qkv)
    ws = torch.empty(B * H * T, dtype=torch.float32, device=qkv.device)
    if dropout is None:
        L.check(L.load().a2f_mha_bwd_train(qkv.data_ptr(), out.data_ptr(), L.ptr(out_f32), dout.data_ptr(), lse.data_ptr(),
                                           dqkv.data_ptr(), _dt(qkv), B, T, H, D, scale, ws.data_ptr(), ws.numel() * 4,
                                           _stream()), "a2f_mha_bwd_train")
        return dqkv
    L.check(L.load().a2f_mha_bwd_train_dropout(qkv.data_ptr(), out.data_ptr(), L.ptr(out_f32), dout.data_ptr(), lse.data_ptr(),
                                               dqkv.data_ptr(), _dt(qkv), B, T, H, D, scale, C.byref(_dropout_args(*dropout)),
                                               ws.data_ptr(), ws.numel() * 4, _stream()), "a2f_mha_bwd_train_dropout")
    return dqkv


def adam_step(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0):
    """fused Adam (+ L2 weight decay) over flat fp32 buffers; `g` fp32, or bf16 as it comes off a bf16 all-reduce.
    `step`: the step count t >= 1 as an int, or a 1-element int32 CUDA tensor holding it (graph-capturable form)."""
    _dev(p, g, m, v)
    if g.numel() != p.numel():
        raise L.A2FError("adam_step: gradient and parameter buffers differ in length")
    if isinstance(step, torch.Tensor):
        _dev(step)
        if step.dtype != torch.int32 or step.numel() != 1 or g.dtype not in (torch.bfloat16, torch.float32):
            raise L.A2FError("adam_step: device step counter must be one int32; gradient fp32 or bf16")
        L.check(L.load().a2f_adam_step_dev(p.data_ptr(), g.data_ptr(), _dt(g), m.data_ptr(), v.data_ptr(), p.numel(), lr, beta1,
                                           beta2, eps, weight_decay, step.data_ptr(), grad_scale, _stream()), "a2f_adam_step_dev")
        return
    fn = L.load().a2f_adam_step_bf16g if g.dtype == torch.bfloat16 else L.load().a2f_adam_step
    if g.dtype not in (torch.bfloat16, torch.float32):
        raise L.A2FError("adam_step: gradient must be fp32 or bf16")
    L.check(fn(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr, beta1, beta2, eps,
               weight_decay, int(step), grad_scale, _stream()), "a2f_adam_step")


def cast_into(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[:] = bf16(x) for contiguous fp32 x / bf16 out of equal length (a2f_cast_f32_to_bf16)."""
    _dev(x, out)
    if x.dtype != torch.float32 or out.dtype != torch.bfloat16 or x.numel() != out.numel() or not (x.is_contiguous() and out.is_contiguous()):
        raise L.A2FError("cast_into: contiguous fp32 -> bf16 of equal length")
    L.check(L.load().a2f_cast_f32_to_bf16(x.data_ptr(), out.data_ptr(), x.numel(), _stream()), "a2f_cast_f32_to_bf16")
    return out


class DecoderTape:
    """Saved activations of one training rollout (a2f_decoder_rollout_train): named [B,T,w] views into one buffer."""

    def __init__(self, B: int, T: int, device):
        lib = L.load()
        self.B, self.T = B, T
        n = len(L.DEC_SAVE_FIELDS)
        offs = [lib.a2f_decoder_save_offset(i) for i in range(n + 1)]
        self.buf = torch.empty(B * T * offs[n], dtype=torch.float32, device=device)
        for i, name in enumerate(L.DEC_SAVE_FIELDS):
            w = offs[i + 1] - offs[i]
            setattr(self, name, self.buf[B * T * offs[i]: B * T * offs[i + 1]].view(B * T, w))
        nbytes = lib.a2f_decoder_workspace_bytes(B, T)
        self.ws = torch.empty((nbytes + 15) // 16 * 4, dtype=torch.float32, device=device)
        self.TMP = self.ws[: B * T * 64].view(B * T, 64)            # v_proj(memory)
        self.CA = self.ws[B * T * 64: 2 * B * T * 64].view(B * T, 64)


def decoder_rollout_train(wstruct, memory, one_hot, period, B, T):
    """-> (D [B,T,64], DecoderTape)"""
    _dev(memory, one_hot)
    tape = DecoderTape(B, T, memory.device)
    D = torch.empty((B, T, 64), dtype=torch.float32, device=memory.device)
    L.check(L.load().a2f_decoder_rollout_train(C.byref(wstruct), memory.data_ptr(), one_hot.data_ptr(), one_hot.shape[1],
                                               period, D.data_ptr(), B, T, tape.ws.data_ptr(), tape.ws.numel() * 4,
                                               tape.buf.data_ptr(), _stream()), "a2f_decoder_rollout_train")
    return D, tape


def decoder_rollout_bwd(wstruct, tape: DecoderTape, gD: torch.Tensor, period: int):
    """-> dict of per-step gradient vectors ([B*T,w] views) + "DSTYLE" [B,64]  (a2f_decoder_rollout_bwd)."""
    _dev(gD)
    lib = L.load()
    B, T = tape.B, tape.T
    n = len(L.DEC_GRAD_FIELDS)
    offs = [lib.a2f_decoder_grad_offset(i) for i in range(n + 1)]
    buf = torch.empty(B * T * offs[n] + B * 64, dtype=torch.float32, device=gD.device)
    nbytes = lib.a2f_decoder_bwd_workspace_bytes(B, T)
    ws = torch.empty((nbytes + 15) // 16 * 4, dtype=torch.float32, device=gD.device)
    L.check(lib.a2f_decoder_rollout_bwd(C.byref(wstruct), tape.buf.data_ptr(), gD.data_ptr(), period, buf.data_ptr(), B, T,
                                        ws.data_ptr(), ws.numel() * 4, _stream()), "a2f_decoder_rollout_bwd")
    out = {"_buf": buf}
    for i, name in enumerate(L.DEC_GRAD_FIELDS):
        w = offs[i + 1] - offs[i]
        out[name] = buf[B * T * offs[i]: B * T * offs[i + 1]].view(B * T, w)
    out["DSTYLE"] = buf[B * T * offs[n]:].view(B, 64)
    return out


def ln64_param_grad(dy, x, dgamma, dbeta):
    _dev(dy, x, dgamma, dbeta)
    L.check(L.load().a2f_ln64_param_grad(dy.data_ptr(), x.data_ptr(), dy.shape[0], dgamma.data_ptr(), dbeta.data_ptr(),
                                         _stream()), "a2f_ln64_param_grad")


def add_strided3(src: torch.Tensor, dst: torch.Tensor, dims, src_strides, dst_strides) -> None:
    """dst[i . dst_strides] += src[i . src_strides] over the 3-D index space `dims` (fp32)."""
    _dev(src, dst)
    if src.dtype != torch.float32 or dst.dtype != torch.float32:
        raise L.A2FError("add_strided3 takes fp32 tensors")
    L.check(L.load().a2f_add_strided3(src.data_ptr(), dst.data_ptr(), *[int(d) for d in dims], *[int(v) for v in src_strides],
                                      *[int(v) for v in dst_strides], _stream()), "a2f_add_strided3")


# ---------------------------------------------------------------------------------------------------------------
# training step of the convolutional models (csrc/conv_train.cu)
# ---------------------------------------------------------------------------------------------------------------
class View:
    """A strided [batches, rows_per_batch, C] window into a padded channels-last fp32 buffer (a2f.h layout convention)."""

    def __init__(self, buf: torch.Tensor, offset: int, C_: int, rows_per_batch: int, ld: int, batch_stride: int, batches: int):
        self.buf, self.offset, self.C, self.rows, self.ld, self.bs, self.batches = buf, offset, C_, rows_per_batch, ld, batch_stride, batches

    @property
    def ptr(self) -> int:
        return self.buf.data_ptr() + 4 * self.offset

    def like(self, buf: torch.Tensor) -> "View":
        return View(buf, self.offset, self.C, self.rows, self.ld, self.bs, self.batches)


def voca_assemble(x: torch.Tensor, one_hot: torch.Tensor) -> torch.Tensor:
    _dev(x, one_hot)
    B = x.shape[0]
    out = torch.empty((B, 17, 37), dtype=torch.float32, device=x.device)
    L.check(L.load().a2f_voca_assemble(x.data_ptr(), one_hot.data_ptr(), one_hot.shape[1], out.data_ptr(), B, _stream()),
            "a2f_voca_assemble")
    return out


def bn_train_stats(v: View, gamma, beta, eps, momentum, running_mean, running_var):
    """-> (mean_rstd [2C], scale_shift [2C]); updates the running statistics in place."""
    _dev(v.buf, gamma, beta, running_mean, running_var)
    mr = torch.empty(2 * v.C, dtype=torch.float32, device=v.buf.device)
    ss = torch.empty(2 * v.C, dtype=torch.float32, device=v.buf.device)
    ws = torch.empty(2 * v.C, dtype=torch.float64, device=v.buf.device)
    L.check(L.load().a2f_bn_train_stats(v.ptr, v.C, v.rows, v.ld, v.bs, v.batches, gamma.data_ptr(), beta.data_ptr(), eps,
                                        momentum, L.ptr(running_mean), L.ptr(running_var), mr.data_ptr(), ss.data_ptr(),
                                        ws.data_ptr(), ws.numel() * 8, _stream()), "a2f_bn_train_stats")
    return mr, ss


def affine_act(src: View, dst: View, scale_shift: Optional[torch.Tensor], act: int) -> None:
    _dev(src.buf, dst.buf, scale_shift)
    sc = scale_shift.data_ptr() if scale_shift is not None else None
    sh = scale_shift.data_ptr() + 4 * src.C if scale_shift is not None else None
    L.check(L.load().a2f_affine_act(src.ptr, dst.ptr, sc, sh, act, src.C, src.rows, src.ld, src.bs, dst.ld, dst.bs,
                                    src.batches, _stream()), "a2f_affine_act")


def bn_train_bwd(dy: View, y_relu: Optional[View], z: View, mean_rstd, gamma, dz: View, dgamma, dbeta) -> None:
    _dev(dy.buf, z.buf, dz.buf, mean_rstd, gamma, dgamma, dbeta)
    for o in (y_relu, z, dz):
        if o is not None and (o.ld, o.bs, o.rows, o.batches, o.C) != (dy.ld, dy.bs, dy.rows, dy.batches, dy.C):
            raise L.A2FError("bn_train_bwd: all views must share one layout")
    ws = torch.empty(2 * dy.C, dtype=torch.float64, device=dy.buf.device)
    L.check(L.load().a2f_bn_train_bwd(dy.ptr, y_relu.ptr if y_relu is not None else None, z.ptr, mean_rstd.data_ptr(),
                                      gamma.data_ptr(), dy.C, dy.rows, dy.ld, dy.bs, dy.batches, dz.ptr, dgamma.data_ptr(),
                                      dbeta.data_ptr(), ws.data_ptr(), ws.numel() * 8, _stream()), "a2f_bn_train_bwd")


# ---------------------------------------------------------------------------------------------------- MFCC extractor
def mfcc_frames(audio: torch.Tensor, win: int, hop: int, n_fft: int, kpad: int, dtype: torch.dtype, gmax: torch.Tensor):
    """audio [B,N] fp32 -> frame matrix [B*F, kpad] fp32 or [B*F, 3*kpad] bf16 split (a2f_mfcc_frames)."""
    _dev(audio, gmax)
    B, N = audio.shape
    F_ = 1 + N // hop
    out = torch.empty((B * F_, kpad if dtype == torch.float32 else 3 * kpad), dtype=dtype, device=audio.device)
    L.check(L.load().a2f_mfcc_frames(audio.data_ptr(), B, N, win, hop, n_fft, kpad, out.data_ptr(), _dt(out), gmax.data_ptr(),
                                     _stream()), "a2f_mfcc_frames")
    return out, F_


def mfcc_mel_db(spec: torch.Tensor, n_freq: int, fb: torch.Tensor, band: torch.Tensor, gmax: torch.Tensor) -> torch.Tensor:
    _dev(spec, fb, band, gmax)
    M, n_mels = spec.shape[0], fb.shape[1]
    db = torch.empty((M, n_mels), dtype=torch.float32, device=spec.device)
    L.check(L.load().a2f_mfcc_mel_db(spec.data_ptr(), spec.stride(0), M, n_freq, fb.data_ptr(), band.data_ptr(), n_mels,
                                     db.data_ptr(), gmax.data_ptr(), _stream()), "a2f_mfcc_mel_db")
    return db


def mfcc_dct_resize(db: torch.Tensor, gmax: torch.Tensor, top_db: float, dct: torch.Tensor, B: int, F_: int,
                    out_dim: int) -> torch.Tensor:
    _dev(db, gmax, dct)
    n_mels, n_mfcc = dct.shape
    out = torch.empty((B, out_dim, n_mfcc), dtype=torch.float32, device=db.device)
    L.check(L.load().a2f_mfcc_dct_resize(db.data_ptr(), gmax.data_ptr(), float(top_db), dct.data_ptr(), B, F_, n_mels, n_mfcc,
                                         out_dim, out.data_ptr(), _stream()), "a2f_mfcc_dct_resize")
    return out
