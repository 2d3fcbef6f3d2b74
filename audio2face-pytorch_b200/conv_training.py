"""Training step of the three convolutional models on the sm_100a kernels: forward that keeps a tape + explicit backward
(ref: torch.autograd over ref:src/model/voca.py:38-49 / ref:src/model/audio2face.py:57-66 / ref:src/model/song2face.py:63-76
inside Lightning's training_step, ref:src/model/lightning_model.py:150-161).

Audio2Mesh and Song2Face run their BatchNorms in TRAIN mode here (batch statistics, running-stat update,
num_batches_tracked += 1), exactly what `model.train()` means in the reference; VOCA has no stochastic or batch-dependent
op, and Song2Face's single-layer LSTMs have no dropout.  The whole training path uses the true-fp32 SIMT GEMMs whatever
the module's precision: VOCA / Audio2Mesh forward convolutions as implicit GEMMs over zero-left-padded channels-last
activations with data gradients as gather-segment GEMMs; Song2Face's convolutions as explicit im2col + GEMM with the
data gradient through the im2col adjoint (a2f_col2im1d); its LSTMs as the input-projection GEMM + the cluster recurrence,
backward through a2f_lstm_bptt.  Weight gradients are transposed-operand GEMMs accumulated straight into `.grad`.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import lib as L
from . import ops

S = L.SIMT_F32
RELU, TANH, NONE = L.ACT_RELU, L.ACT_TANH, L.ACT_NONE


from .training import _grad, collect_grads      # noqa: E402  (gradient sink shared with the FaceFormer backward)


class Pad:
    """Zero-left-padded channels-last activation [nb, L+1, C] (row 0 of every block is the conv's left padding)."""

    def __init__(self, nb: int, L_: int, C_: int, device, buf: Optional[torch.Tensor] = None):
        self.nb, self.L, self.C = nb, L_, C_
        self.buf = buf if buf is not None else torch.zeros((nb, L_ + 1, C_), dtype=torch.float32, device=device)

    def view(self) -> ops.View:
        return ops.View(self.buf, self.C, self.C, self.L, self.C, (self.L + 1) * self.C, self.nb)

    def valid(self) -> torch.Tensor:
        return self.buf.view(-1)[self.C:]

    def zeros_like(self) -> "Pad":
        return Pad(self.nb, self.L, self.C, self.buf.device)


def conv_mat(w: torch.Tensor) -> torch.Tensor:
    """[Co,Ci,kh,kw] with one unit kernel dim -> implicit-GEMM matrix [Co, tap*Ci + ci]."""
    w3 = w.detach().reshape(w.shape[0], w.shape[1], -1)
    return w3.permute(0, 2, 1).reshape(w.shape[0], -1).contiguous()


def conv_k3s2_fwd(xp: Pad, wmat: torch.Tensor, bias: torch.Tensor, act: int) -> Pad:
    Ci, Co, Lo = xp.C, wmat.shape[0], xp.L // 2
    out = Pad(xp.nb, Lo, Co, xp.buf.device)
    ops.gemm(xp.buf, wmat, out.buf, bias=bias, act=act, backend=S, M=xp.nb * Lo, K=3 * Ci, a_row_stride=2 * Ci,
             a_batch_stride=(xp.L + 1) * Ci, rows_per_batch=Lo, ldc=Co, c_batch_stride=(Lo + 1) * Co, c_offset=Co)
    return out


def conv_k3s2_bwd(xp: Pad, dzp: Pad, conv: torch.nn.Module, need_dx: bool) -> Optional[Pad]:
    """dzp: gradient wrt the conv OUTPUT (pre-activation), padded layout with zero padding rows."""
    w = conv.weight
    Co, Ci = w.shape[0], w.shape[1]
    Lo, Lin = dzp.L, xp.L
    dev = xp.buf.device
    nb = xp.nb
    # bias: the padding rows of dzp are zero, so the column sum over the whole buffer is the sum over the valid rows
    ops.colsum(dzp.buf.view(-1, Co), _grad(conv.bias))
    # weight: dW[co, tap*Ci + ci] = sum_{b,t} dz[b,t,co] * xpad[b, 2t + tap, ci]
    dwp = torch.zeros((Co, 3 * Ci), dtype=torch.float32, device=dev)
    ops.gemm_wgrad(dzp.valid(), xp.buf, dwp, backend=S, M=nb * Lo, N=Co, K=Ci, dy_row_stride=Co,
                   dy_batch_stride=(Lo + 1) * Co, x_row_stride=2 * Ci, x_batch_stride=(Lin + 1) * Ci, rows_per_batch=Lo,
                   x_rows=(Lin + 2) // 2, segs=[(0, 0), (0, Ci), (1, 0)])
    ops.add_strided3(dwp, _grad(w), (Co, 3, Ci), (3 * Ci, Ci, 1), (3 * Ci, 1, 3))
    if not need_dx:
        return None
    # data: padded position i = 2t + tap.  even i = 2u: taps 0 (t=u) and 2 (t=u-1); odd i = 2u+1: tap 1 (t=u)
    w3 = w.detach().reshape(Co, Ci * 3)
    even = torch.empty((Ci, 2 * Co), dtype=torch.float32, device=dev)
    ops.transpose_cast(w3, torch.float32, R=Co, Cc=Ci, ld_r=3 * Ci, ld_c=3, offset=2, out=even, ldo=2 * Co, out_offset=0)
    ops.transpose_cast(w3, torch.float32, R=Co, Cc=Ci, ld_r=3 * Ci, ld_c=3, offset=0, out=even, ldo=2 * Co, out_offset=Co)
    odd = ops.transpose_cast(w3, torch.float32, R=Co, Cc=Ci, ld_r=3 * Ci, ld_c=3, offset=1)
    dxp = xp.zeros_like()
    U = Lo + 1
    ops.gemm(dzp.valid(), even, dxp.buf, backend=S, M=nb * U, K=2 * Co, N=Ci, a_row_stride=Co,
             a_batch_stride=(Lo + 1) * Co, rows_per_batch=U, a_rows=Lo, segs=[(-1, 0), (0, 0)], ldc=2 * Ci,
             c_batch_stride=(Lin + 1) * Ci)
    ops.gemm(dzp.valid(), odd, dxp.buf, backend=S, M=nb * Lo, K=Co, N=Ci, a_row_stride=Co, a_batch_stride=(Lo + 1) * Co,
             rows_per_batch=Lo, ldc=2 * Ci, c_batch_stride=(Lin + 1) * Ci, c_offset=Ci)
    return dxp


def linear_bwd(dy: torch.Tensor, x: torch.Tensor, lin_w: torch.nn.Parameter, lin_b: Optional[torch.nn.Parameter], need_dx: bool,
               K: Optional[int] = None, w_cols: Optional[slice] = None) -> Optional[torch.Tensor]:
    """y = x W^T + b backward.  dy [M,N]; x [M, >=K] (row stride may exceed K); W [N, Ktot] (columns w_cols used)."""
    N = dy.shape[1]
    K = int(K if K is not None else x.shape[1])
    gw = _grad(lin_w)
    c0 = w_cols.start if w_cols is not None else 0
    ops.gemm_wgrad(dy, x, gw.view(-1)[c0:], backend=S, N=N, K=K, ldw=gw.stride(0))
    if lin_b is not None:
        ops.colsum(dy, _grad(lin_b))
    if not need_dx:
        return None
    wt = ops.transpose_cast(lin_w.detach(), torch.float32, R=N, Cc=K, ld_r=lin_w.stride(0), offset=c0)     # [K, N]
    dx = torch.empty((dy.shape[0], K), dtype=torch.float32, device=dy.device)
    ops.gemm(dy, wt, dx, backend=S)
    return dx


def _head_bwd(dout: torch.Tensor, z64: torch.Tensor, head: torch.nn.Linear) -> torch.Tensor:
    """out = z[:, :50] W^T + b + template.  z64: [B,64] zero-padded."""
    return linear_bwd(dout, z64, head.weight, head.bias, True, K=head.weight.shape[1])


# ---------------------------------------------------------------------------------------------------------------
# VOCA
# ---------------------------------------------------------------------------------------------------------------
def voca_forward_train(m, x, one_hot, tmpl):
    bs = x.shape[0]
    dev = x.device
    acts: List[Pad] = [Pad(bs, 16, 37, dev, buf=ops.voca_assemble(x, one_hot))]
    for idx in (0, 2, 4, 6):
        conv = m.time_conv[idx]
        acts.append(conv_k3s2_fwd(acts[-1], conv_mat(conv.weight), conv.bias.detach(), RELU))
    feat = acts[-1].buf[:, 1, :]                                  # [bs, 64] (row stride 128)
    fc = m.decoder
    oh8 = one_hot[:, :8].contiguous()
    w0 = fc[0].weight.detach()
    part = torch.empty((bs, 72), dtype=torch.float32, device=dev)     # cat((feat, one_hot8)) @ W0^T as two GEMMs
    ops.gemm(oh8, w0[:, 64:], part, bias=fc[0].bias.detach(), backend=S, K=8)
    f0 = torch.empty((bs, 72), dtype=torch.float32, device=dev)
    ops.gemm(feat, w0, f0, resid=part, backend=S, K=64)
    f1pre = torch.empty((bs, 128), dtype=torch.float32, device=dev)
    ops.gemm(f0, fc[1].weight.detach(), f1pre, bias=fc[1].bias.detach(), backend=S)
    f1 = ops.act_fwd(f1pre, TANH)
    z = torch.zeros((bs, 64), dtype=torch.float32, device=dev)
    ops.gemm(f1, fc[3].weight.detach(), z, bias=fc[3].bias.detach(), backend=S, ldc=64)
    out = m._vertex_head(z, fc[4].weight, fc[4].bias, tmpl, 1, 50)
    return out.view(bs, -1, 3), dict(acts=acts, feat=feat, oh8=oh8, f0=f0, f1pre=f1pre, f1=f1, z=z)


def voca_backward(m, tp: Dict, dout: torch.Tensor) -> None:
    fc = m.decoder
    bs = dout.shape[0]
    dout = dout.reshape(bs, -1)
    dz = _head_bwd(dout, tp["z"], fc[4])
    df1 = linear_bwd(dz, tp["f1"], fc[3].weight, fc[3].bias, True)
    df1pre = ops.act_bwd(df1, tp["f1pre"], TANH)
    df0 = linear_bwd(df1pre, tp["f0"], fc[1].weight, fc[1].bias, True)
    linear_bwd(df0, tp["oh8"], fc[0].weight, fc[0].bias, False, K=8, w_cols=slice(64, 72))
    dfeat = linear_bwd(df0, tp["feat"], fc[0].weight, None, True, K=64, w_cols=slice(0, 64))
    acts = tp["acts"]
    dyp = acts[4].zeros_like()                                    # [bs, 2, 64]: grad wrt the last conv's ReLU output
    dyp.buf[:, 1, :] = dfeat
    for li, idx in zip((3, 2, 1, 0), (6, 4, 2, 0)):
        dzp = Pad(dyp.nb, dyp.L, dyp.C, dyp.buf.device, buf=ops.act_bwd(dyp.buf, acts[li + 1].buf, RELU))   # y > 0 <=> z > 0
        dyp = conv_k3s2_bwd(acts[li], dzp, m.time_conv[idx], need_dx=li > 0)


# ---------------------------------------------------------------------------------------------------------------
# Audio2Mesh
# ---------------------------------------------------------------------------------------------------------------
def _bn_fwd(bn: torch.nn.BatchNorm2d, src: ops.View):
    """train-mode statistics of `src` + running-stat update (momentum None = cumulative average is not used by the
    reference: nn.BatchNorm2d defaults, momentum 0.1)."""
    mr, ss = ops.bn_train_stats(src, bn.weight.detach(), bn.bias.detach(), bn.eps, bn.momentum, bn.running_mean, bn.running_var)
    bn.num_batches_tracked += 1
    for t in (bn.running_mean, bn.running_var):          # written through raw pointers: invalidate derived-weight caches
        torch.autograd.graph.increment_version(t)
    return mr, ss


def a2m_forward_train(m, x, one_hot, tmpl):
    bs = x.shape[0]
    dev = x.device
    CH = m._CH
    tp: Dict = {"ana": [], "art": []}
    cur = Pad(bs * 64, 32, 1, dev, buf=ops.a2m_assemble(x, one_hot).view(bs * 64, 33, 1))
    # ---- formant analysis net: conv along W -> BN -> ReLU (ref audio2face.py:13-29) ----
    for i in range(5):
        conv, bn = m.analysis_net[3 * i], m.analysis_net[3 * i + 1]
        wmat = conv_mat(conv.weight)
        if i < 4:
            z = conv_k3s2_fwd(cur, wmat, conv.bias.detach(), NONE)
            y = z.zeros_like()
        else:                                                      # W: 2 -> 1, lands in the articulation layout [bs,65,256]
            z = Pad(bs, 64, 256, dev)
            ops.gemm(cur.buf, wmat, z.buf, bias=conv.bias.detach(), backend=S, M=bs * 64, K=3 * CH[4], a_row_stride=3 * CH[4],
                     a_batch_stride=64 * 3 * CH[4], rows_per_batch=64, ldc=256, c_batch_stride=65 * 256, c_offset=256)
            y = z.zeros_like()
        mr, ss = _bn_fwd(bn, z.view())
        ops.affine_act(z.view(), y.view(), ss, RELU)
        tp["ana"].append(dict(x=cur, z=z, y=y, mr=mr))
        cur = y
    # ---- articulation net: conv along H ----
    for ci, bi in ((0, 1), (3, 4), (6, 7)):                        # conv -> BN -> ReLU (ref audio2face.py:31-40)
        conv, bn = m.articulation_net[ci], m.articulation_net[bi]
        z = conv_k3s2_fwd(cur, conv_mat(conv.weight), conv.bias.detach(), NONE)
        y = z.zeros_like()
        mr, ss = _bn_fwd(bn, z.view())
        ops.affine_act(z.view(), y.view(), ss, RELU)
        tp["art"].append(dict(x=cur, z=z, y=y, mr=mr))
        cur = y
    bn, conv = m.articulation_net[9], m.articulation_net[10]       # BN -> conv -> ReLU (ref audio2face.py:41-43)
    mr, ss = _bn_fwd(bn, cur.view())
    u = cur.zeros_like()
    ops.affine_act(cur.view(), u.view(), ss, NONE)
    y = conv_k3s2_fwd(u, conv_mat(conv.weight), conv.bias.detach(), RELU)
    tp["art"].append(dict(x=cur, u=u, y=y, mr=mr))
    cur = y                                                        # [bs, 4(+1), 256]
    bn, conv = m.articulation_net[12], m.articulation_net[13]      # BN -> conv(4x1, stride 4) -> ReLU (:44-46)
    mr, ss = _bn_fwd(bn, cur.view())
    u = cur.zeros_like()
    ops.affine_act(cur.view(), u.view(), ss, NONE)
    feat = torch.empty((bs, 256), dtype=torch.float32, device=dev)
    ops.gemm(u.valid(), conv_mat(conv.weight), feat, bias=conv.bias.detach(), act=RELU, backend=S, M=bs, K=1024,
             a_row_stride=5 * 256, rows_per_batch=bs)
    tp["art"].append(dict(x=cur, u=u, mr=mr))
    return output_net_forward(m, feat, one_hot, tmpl, tp), tp


def output_net_forward(m, feat: torch.Tensor, one_hot: torch.Tensor, tmpl: torch.Tensor, tp: Dict) -> torch.Tensor:
    """Output MLP + vertex head shared by Audio2Mesh and Song2Face (ref audio2face.py:49-55,65-66 / song2face.py:74-76):
    cat((feat, one_hot)) -> Linear -> Linear -> Tanh -> Linear -> Linear + template.  feat [bs, 256]; tapes into `tp`."""
    bs = feat.shape[0]
    dev = feat.device
    fc = m.output_net
    w0 = fc[0].weight.detach()
    part = torch.empty((bs, 72), dtype=torch.float32, device=dev)
    ops.gemm(one_hot, w0[:, 256:], part, bias=fc[0].bias.detach(), backend=S, K=m.n_onehot)
    f0 = torch.empty((bs, 72), dtype=torch.float32, device=dev)
    ops.gemm(feat, w0, f0, resid=part, backend=S, K=256)
    f1pre = torch.empty((bs, 128), dtype=torch.float32, device=dev)
    ops.gemm(f0, fc[1].weight.detach(), f1pre, bias=fc[1].bias.detach(), backend=S)
    f1 = ops.act_fwd(f1pre, TANH)
    z = torch.zeros((bs, 64), dtype=torch.float32, device=dev)
    ops.gemm(f1, fc[3].weight.detach(), z, bias=fc[3].bias.detach(), backend=S, ldc=64)
    out = m._vertex_head(z, fc[4].weight, fc[4].bias, tmpl, 1, 50)
    tp.update(feat=feat, one_hot=one_hot, f0=f0, f1pre=f1pre, f1=f1, zhead=z)
    return out.view(bs, -1, 3)


def output_net_backward(m, tp: Dict, dout: torch.Tensor) -> torch.Tensor:
    """Backward of output_net_forward.  feat is the ReLU output of the model's last conv: returns the gradient wrt that
    conv's pre-activation."""
    fc = m.output_net
    bs = dout.shape[0]
    dout = dout.reshape(bs, -1)
    dz = _head_bwd(dout, tp["zhead"], fc[4])
    df1 = linear_bwd(dz, tp["f1"], fc[3].weight, fc[3].bias, True)
    df1pre = ops.act_bwd(df1, tp["f1pre"], TANH)
    df0 = linear_bwd(df1pre, tp["f0"], fc[1].weight, fc[1].bias, True)
    linear_bwd(df0, tp["one_hot"], fc[0].weight, fc[0].bias, False, K=m.n_onehot, w_cols=slice(256, 256 + m.n_onehot))
    dfeat = linear_bwd(df0, tp["feat"], fc[0].weight, None, True, K=256, w_cols=slice(0, 256))
    return ops.act_bwd(dfeat, tp["feat"], RELU)


def _bn_bwd(bn, dy: Pad, y_relu: Optional[Pad], z: Pad, mr) -> Pad:
    dz = z.zeros_like()
    ops.bn_train_bwd(dy.view(), y_relu.view() if y_relu is not None else None, z.view(), mr, bn.weight.detach(), dz.view(),
                     _grad(bn.weight), _grad(bn.bias))
    return dz


def a2m_backward(m, tp: Dict, dout: torch.Tensor) -> None:
    bs = dout.shape[0]
    dev = dout.device
    CH = m._CH
    dfeat = output_net_backward(m, tp, dout)
    # ---- articulation layer 5: BN -> conv(4x1, s4) -> ReLU ----
    a = tp["art"][4]
    conv, bn = m.articulation_net[13], m.articulation_net[12]
    ops.colsum(dfeat, _grad(conv.bias))
    dwp = torch.zeros((256, 1024), dtype=torch.float32, device=dev)
    ops.gemm_wgrad(dfeat, a["u"].valid(), dwp, backend=S, N=256, K=1024, x_row_stride=5 * 256)
    ops.add_strided3(dwp, _grad(conv.weight), (256, 4, 256), (1024, 256, 1), (1024, 1, 4))
    du = a["u"].zeros_like()
    wt = ops.transpose_cast(conv_mat(conv.weight), torch.float32)                      # [1024, 256]
    ops.gemm(dfeat, wt, du.buf, backend=S, ldc=5 * 256, c_offset=256)
    dy = _bn_bwd(bn, du, None, a["x"], a["mr"])
    # ---- articulation layer 4: BN -> conv -> ReLU ----
    a = tp["art"][3]
    conv, bn = m.articulation_net[10], m.articulation_net[9]
    dzp = Pad(dy.nb, dy.L, dy.C, dev, buf=ops.act_bwd(dy.buf, a["y"].buf, RELU))
    du = conv_k3s2_bwd(a["u"], dzp, conv, True)
    dy = _bn_bwd(bn, du, None, a["x"], a["mr"])
    # ---- articulation layers 3..1: conv -> BN -> ReLU ----
    for j, (ci, bi) in zip((2, 1, 0), ((6, 7), (3, 4), (0, 1))):
        a = tp["art"][j]
        dzp = _bn_bwd(m.articulation_net[bi], dy, a["y"], a["z"], a["mr"])
        dy = conv_k3s2_bwd(a["x"], dzp, m.articulation_net[ci], True)
    # ---- analysis layer 5 (W 2 -> 1): a Linear 3*243 -> 256 per (b, h) ----
    a = tp["ana"][4]
    conv, bn = m.analysis_net[12], m.analysis_net[13]
    dzp = _bn_bwd(bn, dy, a["y"], a["z"], a["mr"])
    ops.colsum(dzp.buf.view(-1, 256), _grad(conv.bias))
    Ci = CH[4]
    dwp = torch.zeros((256, 3 * Ci), dtype=torch.float32, device=dev)
    ops.gemm_wgrad(dzp.valid(), a["x"].buf, dwp, backend=S, M=bs * 64, N=256, K=3 * Ci, dy_row_stride=256,
                   dy_batch_stride=65 * 256, x_row_stride=3 * Ci, x_batch_stride=64 * 3 * Ci, rows_per_batch=64)
    ops.add_strided3(dwp, _grad(conv.weight), (256, 3, Ci), (3 * Ci, Ci, 1), (3 * Ci, 1, 3))
    wt = ops.transpose_cast(conv_mat(conv.weight), torch.float32)                      # [3*Ci, 256]
    dy = a["x"].zeros_like()                                                           # [bs*64, 3, Ci]; column 0 = padding
    ops.gemm(dzp.valid(), wt, dy.buf, backend=S, M=bs * 64, K=256, a_row_stride=256, a_batch_stride=65 * 256,
             rows_per_batch=64, ldc=3 * Ci, c_batch_stride=64 * 3 * Ci)
    # ---- analysis layers 4..1 ----
    for i in (3, 2, 1, 0):
        a = tp["ana"][i]
        dzp = _bn_bwd(m.analysis_net[3 * i + 1], dy, a["y"], a["z"], a["mr"])
        dy = conv_k3s2_bwd(a["x"], dzp, m.analysis_net[3 * i], need_dx=i > 0)


# ---------------------------------------------------------------------------------------------------------------
# Song2Face
# ---------------------------------------------------------------------------------------------------------------
_S2F_ENC = ((5, 2), (5, 2), (3, 1), (3, 1), (3, 1))         # (taps, pad) of the vocal-encoder convs (stride 2 along W)


def _rows(buf: torch.Tensor, C_: int) -> ops.View:
    """[rows, ld] activation (C_ live columns) as one BatchNorm batch"""
    buf2 = buf.view(-1, buf.shape[-1])
    return ops.View(buf2, 0, C_, buf2.shape[0], buf2.stride(0), buf2.numel(), 1)


def _conv_fwd(x, outer, ostride, ld, Ci, Li, taps, pad, conv, bn, x_offset=0):
    """Conv(taps, stride 2, pad) over channels-last x[o*ostride + l*ld + c] as im2col + SIMT GEMM, then BN(train) + ReLU
    (bn given) or ReLU -> (y [outer*Lo, ldc], tape entry)"""
    dev = x.device
    Co = conv.weight.shape[0]
    K = taps * Ci
    kpad = (K + 7) // 8 * 8
    Lo = (Li + 2 * pad - taps) // 2 + 1
    ldc = (Co + 3) // 4 * 4
    col = ops.im2col1d(x, outer, ostride, ld, Ci, Li, taps, 2, pad, kpad, False, x_offset=x_offset)
    wmat = conv_mat(conv.weight)                                   # [Co, tap*Ci + ci]
    z = torch.empty((outer * Lo, ldc), dtype=torch.float32, device=dev)
    e = dict(x=x, geom=(outer, ostride, ld, Ci, Li, taps, pad, x_offset), col=col, wmat=wmat, conv=conv, bn=bn, Co=Co, Lo=Lo,
             ldc=ldc)
    if bn is None:
        ops.gemm(col, wmat, z, bias=conv.bias.detach(), act=RELU, backend=S, N=Co, K=K, ldc=ldc)
        e["y"] = z
        return z, e
    ops.gemm(col, wmat, z, bias=conv.bias.detach(), backend=S, N=Co, K=K, ldc=ldc)
    y = torch.empty_like(z)
    zv = _rows(z, Co)
    mr, ss = _bn_fwd(bn, zv)
    ops.affine_act(zv, zv.like(y), ss, RELU)
    e.update(z=z, y=y, mr=mr)
    return y, e


def _bn_relu_bwd(e: Dict, dy: torch.Tensor) -> torch.Tensor:
    """gradient wrt the conv output z of y = ReLU(BN(z)), given dy"""
    Co, bn = e["Co"], e["bn"]
    dz = torch.empty_like(e["z"])
    ops.bn_train_bwd(_rows(dy, Co), _rows(e["y"], Co), _rows(e["z"], Co), e["mr"], bn.weight.detach(), _rows(dz, Co),
                     _grad(bn.weight), _grad(bn.bias))
    return dz


def _conv_bwd(e: Dict, dz: torch.Tensor, need_dx: bool) -> Optional[torch.Tensor]:
    """dz: gradient wrt the conv output [outer*Lo, ldc].  Accumulates dW, db; returns dx laid out like the conv input."""
    outer, ostride, ld, Ci, Li, taps, pad, x_offset = e["geom"]
    conv, col, Co = e["conv"], e["col"], e["Co"]
    K = taps * Ci
    dwp = torch.zeros((Co, K), dtype=torch.float32, device=dz.device)
    ops.gemm_wgrad(dz, col, dwp, backend=S, N=Co, K=K)
    ops.add_strided3(dwp, _grad(conv.weight), (Co, taps, Ci), (K, Ci, 1), (Ci * taps, 1, taps))
    ops.colsum(dz, _grad(conv.bias), cols=Co)
    if not need_dx:
        return None
    wt = ops.transpose_cast(e["wmat"], torch.float32)              # [K, Co]
    dcol = torch.empty_like(col)
    ops.gemm(dz, wt, dcol, backend=S, K=Co)
    return ops.col2im1d(dcol, torch.empty_like(e["x"]), outer, ostride, ld, Ci, Li, taps, 2, pad, x_offset)


def lstm_forward_train(lstm: torch.nn.LSTM, x: torch.Tensor):
    """single-layer batch_first nn.LSTM (hidden 256, zero initial state) on x [B,T,I] -> (h [B,T,256], tape entry)"""
    B, T, I = x.shape
    xp = torch.empty((B * T, 1024), dtype=torch.float32, device=x.device)
    ops.gemm(x.reshape(B * T, I), lstm.weight_ih_l0.detach(), xp, bias=lstm.bias_ih_l0.detach() + lstm.bias_hh_l0.detach(),
             backend=S)
    h, gates, cell = ops.lstm_recurrence_train(xp, lstm.weight_hh_l0.detach(), B, T, 256)
    return h, dict(x=x, h=h, gates=gates, cell=cell)


def lstm_backward(lstm: torch.nn.LSTM, e: Dict, dh: torch.Tensor, need_dx: bool = True) -> Optional[torch.Tensor]:
    """dh [B,T,256] = dL/dh_t from above the layer -> accumulates the four parameter gradients; returns dL/dx [B,T,I]"""
    x, h = e["x"], e["h"]
    B, T, I = x.shape
    H = h.shape[2]
    da = ops.lstm_bptt(dh.contiguous(), e["gates"], e["cell"], lstm.weight_hh_l0.detach()).view(B * T, 4 * H)
    if T > 1:                        # dW_hh = sum_{t>=1} da_t^T h_{t-1}: rows t = 1..T-1 of da against rows 0..T-2 of h
        ops.gemm_wgrad(da, h, _grad(lstm.weight_hh_l0), backend=S, M=B * (T - 1), N=4 * H, K=H, dy_offset=4 * H,
                       dy_row_stride=4 * H, dy_batch_stride=T * 4 * H, x_row_stride=H, x_batch_stride=T * H, rows_per_batch=T - 1)
    ops.gemm_wgrad(da, x.reshape(B * T, I), _grad(lstm.weight_ih_l0), backend=S)
    ops.colsum(da, _grad(lstm.bias_ih_l0))
    ops.colsum(da, _grad(lstm.bias_hh_l0))
    if not need_dx:
        return None
    wt = ops.transpose_cast(lstm.weight_ih_l0.detach(), torch.float32)            # [I, 4H]
    dx = torch.empty((B * T, I), dtype=torch.float32, device=x.device)
    ops.gemm(da, wt, dx, backend=S)
    return dx.view(B, T, I)


def s2f_forward_train(m, x, one_hot, tmpl):
    bs = x.shape[0]
    tp: Dict = {"enc": [], "lstm": [], "reg": []}
    # ---- vocal encoder: conv along W -> BN -> ReLU (ref song2face.py:33-39) ----
    cur = ops.a2m_assemble(x, one_hot)                              # [B,64,33]; column 0 is an unused zero pad
    outer, ostride, ld, Ci, Li, xoff = bs * 64, 33, 1, 1, 32, 1
    for i, (taps, pad) in enumerate(_S2F_ENC):
        seq = m.vocal_encoder_nn[i]
        cur, e = _conv_fwd(cur, outer, ostride, ld, Ci, Li, taps, pad, seq[0], seq[1], x_offset=xoff)
        tp["enc"].append(e)
        ostride, ld, Ci, Li, xoff = e["Lo"] * e["ldc"], e["ldc"], e["Co"], e["Lo"], 0
    # ---- two LSTMs over the channel axis: 256 steps of 64 / 256 features (:68-70) ----
    h = ops.transpose_batched(cur.view(bs, 64, 256))
    for lstm in (m.vocal_encoder_lstm1, m.vocal_encoder_lstm2):
        h, e = lstm_forward_train(lstm, h)
        tp["lstm"].append(e)
    # ---- bilinear 256 -> 32 resize, regression net conv -> BN -> ReLU, last conv -> ReLU (:54-59, :71-73) ----
    cur = ops.song2face_resize(h, 32)                               # [B, 32, 256] channels-last
    outer, ostride, Li = bs, 32 * 256, 32
    for i in range(4):
        seq = m.regression_net[i]
        cur, e = _conv_fwd(cur, outer, ostride, 256, 256, Li, 3, 1 if i < 3 else 0, seq[0], seq[1] if i < 3 else None)
        tp["reg"].append(e)
        ostride, Li = e["Lo"] * 256, e["Lo"]
    return output_net_forward(m, cur, one_hot, tmpl, tp), tp       # cur: [B, 256] (one output row per window)


def s2f_backward(m, tp: Dict, dout: torch.Tensor) -> None:
    bs = dout.shape[0]
    dz = output_net_backward(m, tp, dout)
    for i in (3, 2, 1, 0):
        e = tp["reg"][i]
        if i < 3:
            dz = _bn_relu_bwd(e, dy)
        dy = _conv_bwd(e, dz, need_dx=True)
    dh = ops.song2face_resize_bwd(dy.view(bs, 32, 256), 256)
    dh = lstm_backward(m.vocal_encoder_lstm2, tp["lstm"][1], dh)
    dx = lstm_backward(m.vocal_encoder_lstm1, tp["lstm"][0], dh)   # [B, 256 steps, 64 features]
    dy = ops.transpose_batched(dx)                                 # [B, 64, 256] = the last vocal-encoder layer's rows
    for i in (4, 3, 2, 1, 0):
        e = tp["enc"][i]
        dz = _bn_relu_bwd(e, dy)
        dy = _conv_bwd(e, dz, need_dx=i > 0)


_TRAIN_FNS = {"voca": (voca_forward_train, voca_backward), "audio2mesh": (a2m_forward_train, a2m_backward),
              "song2face": (s2f_forward_train, s2f_backward)}


class ConvModelTrainFn(torch.autograd.Function):
    """Glue to torch.autograd for Voca / Audio2Mesh / Song2Face (same scheme as training.FaceformerTrainFn): every parameter
    is an input of the Function and its gradient an output of backward(), so AccumulateGrad / torch DDP hooks fire per
    parameter."""

    @staticmethod
    def forward(ctx, model, kind, x, one_hot, tmpl, *params):
        out, tape = _TRAIN_FNS[kind][0](model, x, one_hot, tmpl)
        ctx.model, ctx.tape, ctx.kind = model, tape, kind
        return out

    @staticmethod
    def backward(ctx, dout):
        bwd = _TRAIN_FNS[ctx.kind][1]
        with collect_grads(list(ctx.model.parameters())) as sink:
            bwd(ctx.model, ctx.tape, dout.contiguous().float())
        ctx.tape = None
        return (None, None, None, None, None) + sink.grads()

    @staticmethod
    def run(model, kind, x, one_hot, tmpl):
        return ConvModelTrainFn.apply(model, kind, x, one_hot, tmpl, *model.parameters())
