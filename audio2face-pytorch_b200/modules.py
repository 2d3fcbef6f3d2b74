"""Drop-in nn.Modules for the reference's model classes (ref:src/model/lightning_model.py:50-58 get_model):
same class names, constructor signature `Model(n_verts, n_onehot)`, `forward(x, one_hot, template, **kwargs)` /
`predict(...)` signatures, parameter / buffer names, shapes and default initialisation (so a reference checkpoint
loads with strict=True) -- but forward() runs the hand-written sm_100a kernels of liba2f_sm100.so.

The parameter containers are ordinary torch layers that are never called; they exist to own the fp32 master
parameters under the reference's state_dict keys.  Derived copies (bf16 casts, implicit-GEMM layouts, the collapsed
decoder feedback matrix) are caches keyed on the parameters' version counters and are never saved.

precision: "fp32"  -> true-fp32 SIMT kernels (parity target 1e-5 m, BASELINE.json north_star)
           "bf16"  -> tcgen05 tensor-core kernels, bf16 operands / fp32 accumulate (parity target 5e-4 m)
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn as nn

from . import lib as L
from . import ops

_PRECISIONS = ("fp32", "bf16")


class _PackCache:
    """Derived-tensor cache invalidated when any source parameter is modified in place or replaced."""

    def __init__(self):
        self._store: Dict[str, tuple] = {}

    def get(self, key: str, sources, build):
        sig = tuple((s.data_ptr(), s._version, s.device) for s in sources)
        hit = self._store.get(key)
        if hit is not None and hit[0] == sig:
            return hit[1]
        if hit is not None and isinstance(hit[1], dict) and "_refresh" in hit[1] and len(hit[0]) == len(sig) and \
                all(a[0] == b[0] and a[2] == b[2] for a, b in zip(hit[0], sig)):
            # same storage, new contents (an optimizer step): re-derive into the existing buffers -- a handful of
            # launches (ops.PackPlan) instead of ~150 per step, and pointers stay valid for captured graphs.  Only the
            # operands of the sources that changed are re-derived (frozen parameters keep their version counter).
            changed = frozenset(b[0] for a, b in zip(hit[0], sig) if a[1] != b[1])
            hit[1]["_refresh"](changed)
            self._store[key] = (sig, hit[1])
            return hit[1]
        val = build()
        self._store[key] = (sig, val)
        return val

    def clear(self):
        self._store.clear()


class GraphedForward:
    """One forward of a drop-in module captured as a CUDA graph (fixed shapes).  Replaying the graph removes the
    ~100 host-side launches of a FaceFormer forward from the critical path.  Call it like the module; inputs are
    copied into the captured input buffers, the returned tensor is the captured output buffer (overwritten by the
    next call)."""

    def __init__(self, module: "nn.Module", x: torch.Tensor, one_hot: torch.Tensor, template: torch.Tensor, **kwargs):
        self.module = module
        self.kwargs = kwargs
        self.static_in = [x.clone(), one_hot.clone(), template.clone()]
        lib = L.load()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(2):                       # warm-up: weight packing, kernel attributes, allocator pools
                module(*self.static_in, **kwargs)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        n0 = lib.a2f_launch_count()
        with torch.no_grad(), torch.cuda.graph(self.graph):
            self.static_out = module(*self.static_in, **kwargs)
        self.launches_per_replay = int(lib.a2f_launch_count() - n0)

    def __call__(self, x, one_hot, template):
        for dst, src in zip(self.static_in, (x, one_hot, template)):
            if dst.data_ptr() != src.data_ptr():
                dst.copy_(src, non_blocking=True)
        self.graph.replay()
        return self.static_out


class _A2FModule(nn.Module):
    def __init__(self):
        super().__init__()
        self.precision = "fp32"
        self._cache = _PackCache()

    def __call__(self, *args, **kwargs):
        # run on the device of the inputs whatever torch's current device is (a torch module would too): the kernels are
        # launched with raw pointers on the current device's stream
        x = args[0] if args else None
        if isinstance(x, torch.Tensor) and x.is_cuda and x.device.index != torch.cuda.current_device():
            with torch.cuda.device(x.device):
                return super().__call__(*args, **kwargs)
        return super().__call__(*args, **kwargs)

    def graphed(self, x, one_hot, template, **kwargs) -> GraphedForward:
        """Capture forward(x, one_hot, template, **kwargs) for these shapes as a CUDA graph."""
        return GraphedForward(self, x, one_hot, template, **kwargs)

    def set_precision(self, precision: str):
        if precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {_PRECISIONS}")
        self.precision = precision
        return self

    def _backend(self) -> int:
        return L.TCGEN05 if self.precision == "bf16" else L.SIMT_F32

    @staticmethod
    def _need_cuda(*ts):
        for t in ts:
            if not t.is_cuda:
                raise L.A2FError("the a2f_b200 modules run on CUDA (sm_100a) only; there is no CPU fallback")

    @staticmethod
    def _no_grad_guard(*ts):
        if torch.is_grad_enabled() and any(t.requires_grad for t in ts):
            raise L.A2FError("autograd through this module is not available; call it under torch.no_grad()")

    def _head_operand(self, weight: nn.Parameter, k_live: int) -> torch.Tensor:
        """bf16x3 split [V3, 192] of the vertex-head weight (zero-padded to 64 input columns), cached per weight version."""
        def build():
            w = torch.zeros((weight.shape[0], 64), dtype=torch.float32, device=weight.device)
            w[:, :k_live] = weight.detach()
            return ops.split_bf16x3(w, True)
        return self._cache.get("head_bf16x3", (weight,), build)

    def _vertex_head(self, z: torch.Tensor, weight: nn.Parameter, bias: nn.Parameter, template2d: torch.Tensor,
                     rows_per_tmpl: int, k_live: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Shared K11 head: out = z @ W^T + b + template, out [M, V3] fp32.  z: fp32 [M, 64] (columns >= k_live zero).

        bf16 precision runs the tcgen05 GEMM on an error-compensated bf16 split (K' = 192: hi*hi + lo*hi + hi*lo), so
        the HBM-bound head keeps ~2^-16 relative accuracy while using the tensor cores."""
        M, v3 = z.shape[0], weight.shape[0]
        if out is None:
            out = torch.empty((M, v3), dtype=torch.float32, device=z.device)
        if self.precision == "bf16":
            wp = self._head_operand(weight, k_live)
            z3 = ops.split_bf16x3(z, False)
            ops.gemm(z3, wp, out, bias=bias.detach(), tmpl=template2d, rows_per_tmpl=rows_per_tmpl, backend=L.TCGEN05, K=192,
                     alg_K=k_live)
        else:
            ops.gemm(z, weight.detach(), out, bias=bias.detach(), tmpl=template2d, rows_per_tmpl=rows_per_tmpl,
                     backend=L.SIMT_F32, K=k_live)
        return out


# ----------------------------------------------------------------------------------------------------------------
class Voca(_A2FModule):
    """Drop-in for ref:src/model/voca.py:5-52."""

    def __init__(self, n_verts: int, n_onehot: int):
        super().__init__()
        self.n_verts = n_verts
        self.n_onehot = n_onehot
        convs = []
        for cin, cout in ((37, 32), (32, 32), (32, 64), (64, 64)):
            convs += [nn.Conv2d(cin, cout, kernel_size=(3, 1), stride=(2, 1), padding=(1, 0)), nn.ReLU()]
        self.time_conv = nn.Sequential(*convs)
        self.decoder = nn.Sequential(nn.Linear(64 + 8, 72), nn.Linear(72, 128), nn.Tanh(), nn.Linear(128, 50),
                                     nn.Linear(50, n_verts))

    def _weights_struct(self):
        def build():
            w = L.VocaWeights()
            keep = []
            for i, idx in enumerate((0, 2, 4, 6)):
                cw = self.time_conv[idx].weight.detach().contiguous()
                cb = self.time_conv[idx].bias.detach().contiguous()
                keep += [cw, cb]
                w.conv_w[i], w.conv_b[i] = cw.data_ptr(), cb.data_ptr()
            for i, idx in enumerate((0, 1, 3)):
                fw = self.decoder[idx].weight.detach().contiguous()
                fb = self.decoder[idx].bias.detach().contiguous()
                keep += [fw, fb]
                w.fc_w[i], w.fc_b[i] = fw.data_ptr(), fb.data_ptr()
            return w, keep
        srcs = [p for p in self.parameters()]
        return self._cache.get("voca_struct", srcs, build)[0]

    def forward(self, x, one_hot, template, **kwargs):
        self._need_cuda(x, one_hot, template)
        bs = x.size(0)
        x = x.contiguous().float()
        one_hot = one_hot.contiguous().float()
        tmpl = template.reshape(bs, -1).contiguous().float()
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # training step: taped forward + explicit backward kernels (conv_training.py), true-fp32 path
            from . import conv_training
            return conv_training.ConvModelTrainFn.run(self, "voca", x, one_hot, tmpl)
        z = torch.empty((bs, 64), dtype=torch.float32, device=x.device)
        ops.voca_trunk(self._weights_struct(), x, one_hot, z)
        out = self._vertex_head(z, self.decoder[4].weight, self.decoder[4].bias, tmpl, 1, 50)
        return out.view(bs, -1, 3)

    def predict(self, x, one_hot, template, **kwargs):
        return self(x, one_hot, template, **kwargs)


# ----------------------------------------------------------------------------------------------------------------
class Audio2Mesh(_A2FModule):
    """Drop-in for ref:src/model/audio2face.py:5-69 (eval-mode BatchNorm).  The ten convs are implicit GEMMs over
    zero-left-padded channels-last activations (csrc/a2m.cu); BatchNorms that follow a conv are folded into the packed
    weights, the two that precede a conv run as a per-channel affine pass."""

    _CH = (1, 72, 108, 162, 243, 256)

    def __init__(self, n_verts: int, n_onehot: int):
        super().__init__()
        self.n_verts = n_verts
        self.n_onehot = n_onehot
        ana = []
        for i in range(5):
            ana += [nn.Conv2d(self._CH[i], self._CH[i + 1], kernel_size=(1, 3), stride=(1, 2), padding=(0, 1)),
                    nn.BatchNorm2d(self._CH[i + 1]), nn.ReLU()]
        self.analysis_net = nn.Sequential(*ana)
        art = []
        for _ in range(3):
            art += [nn.Conv2d(256, 256, kernel_size=(3, 1), stride=(2, 1), padding=(1, 0)), nn.BatchNorm2d(256), nn.ReLU()]
        art += [nn.BatchNorm2d(256), nn.Conv2d(256, 256, kernel_size=(3, 1), stride=(2, 1), padding=(1, 0)), nn.ReLU(),
                nn.BatchNorm2d(256), nn.Conv2d(256, 256, kernel_size=(4, 1), stride=(4, 1)), nn.ReLU()]
        self.articulation_net = nn.Sequential(*art)
        self.output_net = nn.Sequential(nn.Linear(256 + n_onehot, 72), nn.Linear(72, 128), nn.Tanh(), nn.Linear(128, 50),
                                        nn.Linear(50, n_verts))

    @staticmethod
    def _bn_affine(bn: nn.BatchNorm2d):
        s = bn.weight.detach() / torch.sqrt(bn.running_var.detach() + bn.eps)
        return s, bn.bias.detach() - bn.running_mean.detach() * s

    def _packed(self):
        def build():
            def conv_mat(conv, taps_dim):       # [Co,Ci,kh,kw] -> [Co, tap*Ci + ci]
                w = conv.weight.detach()
                w = w[:, :, 0, :] if taps_dim == 3 else w[:, :, :, 0]
                return w.permute(0, 2, 1).reshape(w.shape[0], -1)

            P = {"ana": [], "art": []}
            for i in range(5):
                conv, bn = self.analysis_net[3 * i], self.analysis_net[3 * i + 1]
                s, t = self._bn_affine(bn)
                P["ana"].append(((conv_mat(conv, 3) * s[:, None]).contiguous(), (conv.bias.detach() * s + t).contiguous()))
            for ci, bi in ((0, 1), (3, 4), (6, 7)):
                conv, bn = self.articulation_net[ci], self.articulation_net[bi]
                s, t = self._bn_affine(bn)
                P["art"].append(((conv_mat(conv, 2) * s[:, None]).contiguous(), (conv.bias.detach() * s + t).contiguous()))
            for bi, ci in ((9, 10), (12, 13)):
                s, t = self._bn_affine(self.articulation_net[bi])
                conv = self.articulation_net[ci]
                P["art"].append((conv_mat(conv, 2).contiguous(), conv.bias.detach().contiguous(), s.contiguous(), t.contiguous()))
            return P
        srcs = list(self.parameters()) + [b for b in self.buffers()]
        return self._cache.get("a2m", srcs, build)

    def _packed_tc(self):
        """Tensor-core operands of the conv stack: BN-folded weights [Cout, taps*Cin] zero-padded to Kpad (multiple of
        64) and split hi|hi|lo into bf16 (ops.split_bf16x3) -- the partner of ops.im2col1d_split's hi|lo|hi rows."""
        def build():
            P = self._packed()
            out = {"ana": [], "art": []}

            def split(w):
                kpad = (w.shape[1] + 63) // 64 * 64
                wp = torch.zeros((w.shape[0], kpad), dtype=torch.float32, device=w.device)
                wp[:, :w.shape[1]] = w
                return ops.split_bf16x3(wp, True), kpad
            for w, b in P["ana"]:
                out["ana"].append(split(w) + (b,))
            for ent in P["art"]:
                out["art"].append(split(ent[0]) + tuple(ent[1:]))
            return out
        srcs = list(self.parameters()) + [b for b in self.buffers()]
        return self._cache.get("a2m_tc", srcs, build)

    def _trunk_tc(self, x, one_hot, bs):
        """conv stack on tcgen05 (precision "bf16"): per layer one im2col (fp32 -> bf16 hi|lo|hi split, padding and a
        preceding BatchNorm applied on the fly) and one GEMM with the bias + ReLU epilogue; activations stay fp32."""
        P = self._packed_tc()
        dev = x.device
        T = L.TCGEN05
        cur = ops.a2m_assemble(x, one_hot)                                   # [B,64,33], column 0 is a zero pad (unused here)
        outer, ostride, ld, Ci, Li, xoff = bs * 64, 33, 1, 1, 32, 1
        for i in range(5):                                                   # formant analysis net: conv along W
            w3, kpad, b = P["ana"][i]
            Co = self._CH[i + 1]
            a3 = ops.im2col1d_split(cur, outer, ostride, ld, Ci, Li, 3, 2, 1, kpad, x_offset=xoff)
            Lo = Li // 2
            ldc = (Co + 3) // 4 * 4
            out = torch.empty((outer * Lo, ldc), dtype=torch.float32, device=dev)
            ops.gemm(a3, w3, out, bias=b, act=L.ACT_RELU, backend=T, N=Co, ldc=ldc)
            cur, ostride, ld, Ci, Li, xoff = out, Lo * ldc, ldc, Co, Lo, 0
        outer, ostride, Li = bs, 64 * 256, 64                                # [B*64, 1, 256] is [B, 64, 256]
        for j in range(5):                                                   # articulation net: conv along H
            ent = P["art"][j]
            w3, kpad, b = ent[0], ent[1], ent[2]
            sc, sh = (ent[3], ent[4]) if len(ent) > 3 else (None, None)
            taps, stride, pad = (3, 2, 1) if j < 4 else (4, 4, 0)
            a3 = ops.im2col1d_split(cur, outer, ostride, 256, 256, Li, taps, stride, pad, kpad, scale=sc, shift=sh)
            Lo = (Li + 2 * pad - taps) // stride + 1
            out = torch.empty((outer * Lo, 256), dtype=torch.float32, device=dev)
            ops.gemm(a3, w3, out, bias=b, act=L.ACT_RELU, backend=T)
            cur, ostride, Li = out, Lo * 256, Lo
        return cur                                                           # [B, 256]

    def forward(self, x, one_hot, template, **kwargs):
        self._need_cuda(x, one_hot, template)
        bs = x.size(0)
        dev = x.device
        x = x.contiguous().float()
        one_hot = one_hot.contiguous().float()
        tmpl = template.reshape(bs, -1).contiguous().float()
        grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if self.training:
            # model.train(): each BatchNorm in train() uses batch statistics and updates its running stats, one put in
            # eval() uses its running stats and leaves them alone (conv_training.py)
            from . import conv_training
            if grad:
                return conv_training.ConvModelTrainFn.run(self, "audio2mesh", x, one_hot, tmpl)
            return conv_training.a2m_forward_train(self, x, one_hot, tmpl)[0]
        if grad:
            raise L.A2FError("Audio2Mesh: gradients in eval() mode are not built; run under torch.no_grad(), or, to train "
                             "with frozen BatchNorm statistics, call model.train() and then .eval() on the BatchNorm2d "
                             "layers (ConvModelTrainer(freeze_bn=True) does this) -- the same arithmetic for this model")
        P = self._packed()
        S = L.SIMT_F32
        if self.precision == "bf16":
            feat = self._trunk_tc(x, one_hot, bs)
            return self._output_net(feat, one_hot, tmpl, bs)
        cur = ops.a2m_assemble(x, one_hot)                                   # [B,64,33] (C=1)
        Wi, Ci = 32, 1
        for i in range(5):                                                   # formant analysis net, conv along W
            Co, Wo = self._CH[i + 1], Wi // 2
            w, b = P["ana"][i]
            if i < 4:
                out = torch.zeros((bs, 64, Wo + 1, Co), dtype=torch.float32, device=dev)
                ops.gemm(cur, w, out, bias=b, act=L.ACT_RELU, backend=S, M=bs * 64 * Wo, K=3 * Ci, a_row_stride=2 * Ci,
                         a_batch_stride=(Wi + 1) * Ci, rows_per_batch=Wo, ldc=Co, c_batch_stride=(Wo + 1) * Co, c_offset=Co)
            else:                                                            # W: 2 -> 1, lands in the articulation layout
                out = torch.zeros((bs, 65, 256), dtype=torch.float32, device=dev)
                ops.gemm(cur, w, out, bias=b, act=L.ACT_RELU, backend=S, M=bs * 64, K=3 * Ci, a_row_stride=3 * Ci,
                         a_batch_stride=64 * 3 * Ci, rows_per_batch=64, ldc=256, c_batch_stride=65 * 256, c_offset=256)
            cur, Wi, Ci = out, Wo, Co
        H = 64
        for j in range(4):                                                   # articulation net, conv along H
            Ho = H // 2
            if j < 3:
                w, b = P["art"][j]
            else:
                w, b, s, t = P["art"][3]
                ops.channel_affine(cur, 256, s, t, 256, H, 256, (H + 1) * 256, bs)     # BN before conv (padding stays 0)
            out = torch.zeros((bs, Ho + 1, 256), dtype=torch.float32, device=dev)
            ops.gemm(cur, w, out, bias=b, act=L.ACT_RELU, backend=S, M=bs * Ho, K=768, a_row_stride=512,
                     a_batch_stride=(H + 1) * 256, rows_per_batch=Ho, ldc=256, c_batch_stride=(Ho + 1) * 256, c_offset=256)
            cur, H = out, Ho
        w, b, s, t = P["art"][4]
        ops.channel_affine(cur, 256, s, t, 256, 4, 256, 5 * 256, bs)
        feat = torch.empty((bs, 256), dtype=torch.float32, device=dev)
        ops.gemm(cur.view(-1)[256:], w, feat, bias=b, act=L.ACT_RELU, backend=S, M=bs, K=1024, a_row_stride=5 * 256,
                 rows_per_batch=bs)
        return self._output_net(feat, one_hot, tmpl, bs)

    def _output_net(self, feat, one_hot, tmpl, bs):
        fc = self.output_net
        # cat((feat, one_hot)) -> Linear -> Linear -> Tanh -> Linear in one launch (a2f_a2m_mlp), then the shared vertex head
        z = ops.a2m_mlp(feat, one_hot, fc[0], fc[1], fc[3], ldz=64)
        out = self._vertex_head(z, fc[4].weight, fc[4].bias, tmpl, 1, 50)
        return out.view(bs, -1, 3)

    def predict(self, x, one_hot, template, **kwargs):
        return self(x, one_hot, template, **kwargs)


# ----------------------------------------------------------------------------------------------------------------
class Song2Face(_A2FModule):
    """Drop-in for ref:src/model/song2face.py:5-72 (registry entry "song2face", ref:src/model/lightning_model.py:50-58).
    Same sub-module names, so the state_dict keys (and their order) are the reference's.  eval(): the inference path below
    (eval-mode BatchNorm).  train(): the training step of conv_training.py (batch-statistics BatchNorm, LSTM
    backpropagation through time in a2f_lstm_bptt), like Audio2Mesh.

    Every convolution is an explicit im2col (csrc/a2m.cu) + a2f_gemm with the folded BatchNorm / bias / ReLU epilogue; the
    two LSTMs run over the CHANNEL axis like the reference (256 steps of 64 / 256 features): input projections of all steps
    as one GEMM, the recurrence in a2f_lstm_recurrence (csrc/song2face.cu, fp32); the bilinear 256 -> 32 resize writes the
    channels-last layout the regression convs read; the output MLP and vertex head are Audio2Mesh's.  precision "fp32":
    SIMT GEMMs (1e-5 parity path); "bf16": tcgen05 GEMMs on the error-compensated bf16x3 split."""

    _CH = (1, 72, 108, 162, 243, 256)

    def __init__(self, n_verts: int, n_onehot: int):
        super().__init__()
        self.n_verts = n_verts
        self.n_onehot = n_onehot

        def conv_bn(ci, co, k, st, pad, bn=True):
            mods = [nn.Conv2d(ci, co, k, st, pad)]
            if bn:
                mods.append(nn.BatchNorm2d(co))
            mods.append(nn.ReLU())
            return nn.Sequential(*mods)

        self.vocal_encoder_nn = nn.Sequential(
            conv_bn(1, 72, (1, 5), (1, 2), (0, 2)), conv_bn(72, 108, (1, 5), (1, 2), (0, 2)),
            conv_bn(108, 162, (1, 3), (1, 2), (0, 1)), conv_bn(162, 243, (1, 3), (1, 2), (0, 1)),
            conv_bn(243, 256, (1, 3), (1, 2), (0, 1)))
        self.vocal_encoder_lstm1 = nn.LSTM(64, 256, 1, bidirectional=False, batch_first=True)
        self.vocal_encoder_lstm2 = nn.LSTM(256, 256, 1, bidirectional=False, batch_first=True)
        self.output_net = nn.Sequential(nn.Linear(256 + n_onehot, 72), nn.Linear(72, 128), nn.Tanh(), nn.Linear(128, 50),
                                        nn.Linear(50, n_verts))
        self.regression_net = nn.Sequential(
            conv_bn(256, 256, (3, 1), (2, 1), (1, 0)), conv_bn(256, 256, (3, 1), (2, 1), (1, 0)),
            conv_bn(256, 256, (3, 1), (2, 1), (1, 0)), conv_bn(256, 256, (3, 1), (2, 1), (0, 0), False))

    def _packed(self):
        bf = self.precision == "bf16"

        def build():
            def operand(w2d):                       # [N, K] fp32 -> K padded to 64, bf16x3 split on the tensor-core path
                kpad = (w2d.shape[1] + 63) // 64 * 64
                wp = torch.zeros((w2d.shape[0], kpad), dtype=torch.float32, device=w2d.device)
                wp[:, :w2d.shape[1]] = w2d
                return (ops.split_bf16x3(wp, True) if bf else wp), kpad

            def conv_entry(seq, taps_dim):
                conv = seq[0]
                w = conv.weight.detach()
                w = w[:, :, 0, :] if taps_dim == 3 else w[:, :, :, 0]
                mat = w.permute(0, 2, 1).reshape(w.shape[0], -1)             # [Co, tap*Ci + ci]
                b = conv.bias.detach()
                if isinstance(seq[1], nn.BatchNorm2d):
                    s_, t_ = Audio2Mesh._bn_affine(seq[1])
                    mat, b = mat * s_[:, None], b * s_ + t_
                return operand(mat.contiguous()) + (b.contiguous(),)

            P = {"enc": [conv_entry(seq, 3) for seq in self.vocal_encoder_nn],
                 "reg": [conv_entry(seq, 2) for seq in self.regression_net], "lstm": []}
            for lstm in (self.vocal_encoder_lstm1, self.vocal_encoder_lstm2):
                w_ih, kpad = operand(lstm.weight_ih_l0.detach())
                P["lstm"].append((w_ih, kpad, (lstm.bias_ih_l0.detach() + lstm.bias_hh_l0.detach()).contiguous(),
                                  lstm.weight_hh_l0.detach().t().contiguous(), lstm.weight_hh_l0.detach().contiguous()))
            return P
        srcs = list(self.parameters()) + [b for b in self.buffers()]
        return self._cache.get("s2f_" + self.precision, srcs, build)

    def _conv(self, cur, outer, ostride, ld, Ci, Li, taps, stride, pad, ent, Co, x_offset=0):
        """one conv (+ folded BN) + ReLU over channels-last fp32 [outer, Li, Ci] -> ([outer*Lo, ldc] fp32, Lo, ldc)"""
        bf = self.precision == "bf16"
        w, kpad, b = ent
        a = ops.im2col1d(cur, outer, ostride, ld, Ci, Li, taps, stride, pad, kpad, bf, x_offset=x_offset)
        Lo = (Li + 2 * pad - taps) // stride + 1
        ldc = (Co + 3) // 4 * 4
        out = torch.empty((outer * Lo, ldc), dtype=torch.float32, device=cur.device)
        ops.gemm(a, w, out, bias=b, act=L.ACT_RELU, backend=self._backend(), N=Co, ldc=ldc)
        return out, Lo, ldc

    def forward(self, x, one_hot, template, **kwargs):
        self._need_cuda(x, one_hot, template)
        bs = x.size(0)
        x = x.contiguous().float()
        one_hot = one_hot.contiguous().float()
        tmpl = template.reshape(bs, -1).contiguous().float()
        grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if self.training:
            # model.train(): each BatchNorm in train() uses batch statistics and updates its running stats, one put in
            # eval() uses its running stats; true-fp32 convolutions and LSTMs whatever the precision, the vertex head
            # follows it as for Audio2Mesh (conv_training.py)
            from . import conv_training
            if grad:
                return conv_training.ConvModelTrainFn.run(self, "song2face", x, one_hot, tmpl)
            return conv_training.s2f_forward_train(self, x, one_hot, tmpl)[0]
        if grad:
            raise L.A2FError("Song2Face: gradients in eval() mode are not built; run under torch.no_grad(), or, to train "
                             "with frozen BatchNorm statistics, call model.train() and then .eval() on the BatchNorm2d "
                             "layers (ConvModelTrainer(freeze_bn=True) does this) -- the same arithmetic for this model")
        P = self._packed()
        bf = self.precision == "bf16"
        cur = ops.a2m_assemble(x, one_hot)                                   # [B,64,33]; column 0 is an unused zero pad
        outer, ostride, ld, Ci, Li, xoff = bs * 64, 33, 1, 1, 32, 1
        for i, (taps, pad) in enumerate(((5, 2), (5, 2), (3, 1), (3, 1), (3, 1))):     # vocal encoder, conv along W
            Co = self._CH[i + 1]
            cur, Lo, ldc = self._conv(cur, outer, ostride, ld, Ci, Li, taps, 2, pad, P["enc"][i], Co, x_offset=xoff)
            ostride, ld, Ci, Li, xoff = Lo * ldc, ldc, Co, Lo, 0
        h = ops.transpose_batched(cur.view(bs, 64, 256))                     # [B, steps = 256 channels, features = 64]
        for w_ih, kpad, bias, whh_t, whh in P["lstm"]:
            a2 = h.view(bs * 256, -1)
            if a2.shape[1] != kpad:                                          # features padded to the packed K
                ap = torch.zeros((a2.shape[0], kpad), dtype=torch.float32, device=a2.device)
                ap[:, :a2.shape[1]] = a2
                a2 = ap
            a_op = ops.split_bf16x3(a2, False) if bf else a2
            xp = torch.empty((bs * 256, 1024), dtype=torch.float32, device=x.device)
            ops.gemm(a_op, w_ih, xp, bias=bias, backend=self._backend())
            h = ops.lstm_recurrence(xp, whh_t, bs, 256, 256, whh=whh)        # [B, 256, 256]
        cur = ops.song2face_resize(h, 32)                                    # [B, 32, 256] channels-last (C = LSTM step)
        outer, ostride, Li = bs, 32 * 256, 32
        for i in range(4):                                                   # regression net, conv along the resized axis
            cur, Lo, _ = self._conv(cur, outer, ostride, 256, 256, Li, 3, 2, 1 if i < 3 else 0, P["reg"][i], 256)
            ostride, Li = Lo * 256, Lo
        fc = self.output_net
        z = ops.a2m_mlp(cur, one_hot, fc[0], fc[1], fc[3], ldz=64)
        out = self._vertex_head(z, fc[4].weight, fc[4].bias, tmpl, 1, 50)
        return out.view(bs, -1, 3)

    def predict(self, x, one_hot, template, **kwargs):
        return self(x, one_hot, template, **kwargs)


# ----------------------------------------------------------------------------------------------------------------
class _Box(nn.Module):
    """Plain namespace module: owns parameters / sub-modules under reference-compatible names, never called."""


class _FeatureEncoderBox(_Box):
    """`audio_encoder.feature_extractor`: the freezing API of HF's Wav2Vec2FeatureEncoder."""

    def __init__(self):
        super().__init__()
        self._requires_grad = True

    def _freeze_parameters(self):
        for param in self.parameters():
            param.requires_grad = False
        self._requires_grad = False


class _Wav2Vec2Box(_Box):
    """`audio_encoder`: the freezing API of HF's Wav2Vec2Model (the reference's FaceFormer calls it in its constructor
    when it fine-tunes)."""

    def freeze_feature_encoder(self):
        """Stop the gradient computation of the conv feature encoder (7 conv weights, GroupNorm gamma / beta); the
        training backward then stops above it (training.grad_plan)."""
        self.feature_extractor._freeze_parameters()


def _w2v_param_tree() -> nn.Module:
    """Parameter container with the state_dict keys of the reference's Wav2Vec2Model subclass
    (ref:src/model/wav2vec.py:87; transformers Wav2Vec2Config() base architecture, SURVEY.md App. B.3)."""
    enc = _Wav2Vec2Box()
    enc.masked_spec_embed = nn.Parameter(torch.empty(768).uniform_())
    fe = _FeatureEncoderBox()
    layers = []
    for i, k in enumerate((10, 3, 3, 3, 3, 2, 2)):
        lay = _Box()
        lay.conv = nn.Conv1d(1 if i == 0 else 512, 512, kernel_size=k, stride=5 if i == 0 else 2, bias=False)
        if i == 0:
            lay.layer_norm = nn.GroupNorm(num_groups=512, num_channels=512, affine=True)
        layers.append(lay)
    fe.conv_layers = nn.ModuleList(layers)
    enc.feature_extractor = fe
    fp = _Box()
    fp.layer_norm = nn.LayerNorm(512, eps=1e-5)
    fp.projection = nn.Linear(512, 768)
    enc.feature_projection = fp
    e = _Box()
    pc = _Box()
    pc.conv = nn.utils.parametrizations.weight_norm(nn.Conv1d(768, 768, kernel_size=128, padding=64, groups=16),
                                                    name="weight", dim=2)
    e.pos_conv_embed = pc
    e.layer_norm = nn.LayerNorm(768, eps=1e-5)
    blocks = []
    for _ in range(12):
        blk = _Box()
        att = _Box()
        for nm in ("k_proj", "v_proj", "q_proj", "out_proj"):
            setattr(att, nm, nn.Linear(768, 768))
        blk.attention = att
        blk.layer_norm = nn.LayerNorm(768, eps=1e-5)
        ff = _Box()
        ff.intermediate_dense = nn.Linear(768, 3072)
        ff.output_dense = nn.Linear(3072, 768)
        blk.feed_forward = ff
        blk.final_layer_norm = nn.LayerNorm(768, eps=1e-5)
        blocks.append(blk)
    e.layers = nn.ModuleList(blocks)
    enc.encoder = e
    return enc


class PeriodicPositionalEncoding(nn.Module):
    """Buffer-compatible stand-in for ref:src/model/faceformer.py:70-88 (`pe` [1, (max_seq_len//period+1)*period, d]);
    the decoder kernel indexes row (position mod period) directly, so there is no 600-frame cap."""

    def __init__(self, d_model, dropout=0.1, period=25, max_seq_len=600):
        super().__init__()
        import math
        pe = torch.zeros(period, d_model)
        position = torch.arange(0, period, dtype=torch.float).unsqueeze(1)
        div_term = torch.exp(torch.arange(0, d_model, 2).float() * (-math.log(10000.0) / d_model))
        pe[:, 0::2] = torch.sin(position * div_term)
        pe[:, 1::2] = torch.cos(position * div_term)
        self.register_buffer("pe", pe.unsqueeze(0).repeat(1, (max_seq_len // period) + 1, 1))


class Faceformer(_A2FModule):
    """Drop-in for ref:src/model/faceformer.py:91-191 (inference; eval-mode semantics: dropout / LayerDrop /
    SpecAugment inactive).  Extensions over the reference, all opt-in: batches of B utterances [B,N] (the reference is
    batch-1 only, SURVEY.md fact 0.4), `fps` other than the hard-coded 60 (fact 0.9), clips longer than 600 frames
    (fact 0.8)."""

    def __init__(self, n_verts: int, n_onehot: int):
        super().__init__()
        self.feature_dim = 64
        self.n_onehot = n_onehot
        # training forward only: apply wav2vec2's SpecAugment time masking (ref:src/model/wav2vec.py:149-162) with the
        # reference's host-side numpy draws (spec_augment.py).  None = follow self.training like the reference does;
        # True / False force it.
        self.spec_augment = None
        # training forward only (train() mode, training.forward_train): the wav2vec2 encoder's train-mode dropout and
        # LayerDrop (HF modeling_wav2vec2.py).  False (default) = eval arithmetic.  True applies, with the probabilities of
        # dropout_p, dropout after the feature projection ("feat_proj"), after encoder.layer_norm and on both residual
        # branches of every layer ("hidden"), on the attention probabilities ("attention"), on the FFN activation
        # ("activation"), and skips whole layers ("layerdrop").  The decoder / PPE dropout is not applied.  A no-grad
        # forward is the inference path and stays eval arithmetic.  The defaults are the 960h checkpoint config the
        # reference loads; "feat_proj" = 0.1 is from SURVEY.md A.4, which gives it from memory (not verifiable offline).
        self.encoder_dropout = False
        self.dropout_p = {"hidden": 0.1, "attention": 0.1, "activation": 0.1, "feat_proj": 0.1, "layerdrop": 0.1}
        # Philox key of the dropout masks and seed of the LayerDrop draws (include/a2f.h); None = drawn from torch's default
        # generator at first use; FaceformerTrainer gives every replica rank 0's seed.
        self.dropout_seed = None
        # bf16 inference, 32 / 64 / 128 utterances: the vertex head runs concurrently with the decoder rollout on the SMs the
        # rollout leaves idle (ops.rollout_and_head_stream); False = rollout, then head
        self.stream_head = True
        self.dataset = "vocaset"
        self.period = 60
        self.fps = 60
        self.vertice_dim = n_verts
        self.audio_encoder = _w2v_param_tree()
        self.audio_feature_map = nn.Linear(768, self.feature_dim)
        self.vertice_map = nn.Linear(self.vertice_dim, self.feature_dim)
        self.PPE = PeriodicPositionalEncoding(self.feature_dim, period=self.period)
        layer = nn.TransformerDecoderLayer(d_model=self.feature_dim, nhead=4, dim_feedforward=2 * self.feature_dim,
                                           batch_first=True)
        self.transformer_decoder = nn.TransformerDecoder(layer, num_layers=1)
        self.vertice_map_r = nn.Linear(self.feature_dim, self.vertice_dim)
        self.obj_vector = nn.Linear(self.n_onehot, self.feature_dim, bias=False)
        for p in (self.vertice_map_r.weight, self.vertice_map_r.bias, self.vertice_map.weight, self.vertice_map.bias):
            nn.init.constant_(p, 0)        # ref:faceformer.py:132-135

    # -- derived weights --------------------------------------------------------------------------------------
    def _packed(self):
        bf = self.precision == "bf16"
        dt = torch.bfloat16 if bf else torch.float32
        ae = self.audio_encoder

        def build():
            P = {}
            dev = self.audio_feature_map.weight.device
            plan = ops.PackPlan(dev)
            new = lambda *shape: torch.empty(shape, dtype=dt, device=dev)            # noqa: E731
            cl = ae.feature_extractor.conv_layers
            P["conv0_w"] = cl[0].conv.weight.detach().reshape(512, 10).contiguous()
            convs = []
            for i, k in zip(range(1, 7), (3, 3, 3, 3, 2, 2)):
                w = cl[i].conv.weight.detach()                      # [co, ci, k] -> implicit-GEMM layout [co, tap*ci]
                o = new(512, k * 512)
                for tap in range(k):
                    plan.add(w, o, 512, 512, 512 * k, k, k * 512, 1, src_off=tap, dst_off=tap * 512)
                convs.append(o)
            P["convs"] = convs

            def cast(t):
                t = t.detach()
                if not bf:
                    return t.contiguous()                           # fp32 path reads the masters in place
                o = new(*t.shape)
                plan.cast(t, o)
                return o

            P["proj_w"] = cast(ae.feature_projection.projection.weight)
            pz = ae.encoder.pos_conv_embed.conv.parametrizations.weight
            P["pos_w"] = ops.pack_posconv_weight(pz.original0.detach().reshape(-1), pz.original1.detach(), dt)
            lay = []
            for blk in ae.encoder.layers:
                a = blk.attention
                qkv_w = new(2304, 768)
                qkv_b = torch.empty(2304, dtype=torch.float32, device=dev)
                for j, lin in enumerate((a.q_proj, a.k_proj, a.v_proj)):
                    plan.cast(lin.weight.detach(), qkv_w, dst_off=j * 768 * 768)
                    plan.add(lin.bias.detach(), qkv_b, 1, 768, 768, 1, 768, 1, dst_off=j * 768)
                lay.append({
                    "qkv_w": qkv_w, "qkv_b": qkv_b,
                    "o_w": cast(a.out_proj.weight),
                    "f1_w": cast(blk.feed_forward.intermediate_dense.weight),
                    "f2_w": cast(blk.feed_forward.output_dense.weight),
                })
            P["layers"] = lay
            P["afm_w"] = cast(self.audio_feature_map.weight)
            # cross-attention with the diagonal memory mask is out_proj(v_proj(audio_feature_map(h))): three Linear layers in a
            # row, folded (fp64) into ONE [64, 768] operand so that the encoder states go straight to the vectors the decoder
            # kernel adds (a2f_decoder_rollout_ca); re-derived by fold_ca() with the other packed operands
            ca_w = torch.empty((64, 768), dtype=dt, device=dev)
            ca_b = torch.empty((64,), dtype=torch.float32, device=dev)
            P["ca_w"], P["ca_b"] = ca_w, ca_b

            def fold_ca():
                ca_mod = self.transformer_decoder.layers[0].multihead_attn
                ops.pack_cross_attention(ca_mod.in_proj_weight.detach(), ca_mod.in_proj_bias.detach(),
                                         ca_mod.out_proj.weight.detach(), ca_mod.out_proj.bias.detach(),
                                         self.audio_feature_map.weight.detach(), self.audio_feature_map.bias.detach(), ca_w, ca_b)
            wc = torch.empty((64, 64), dtype=torch.float32, device=dev)
            bc = torch.empty((64,), dtype=torch.float32, device=dev)
            P["fb"] = (wc, bc)
            # feedback and next-token in-projection applied as one matvec by the rollout kernels (a2f_pack_decoder_fold)
            fold_w = torch.empty((192, 64), dtype=torch.float32, device=dev)
            fold_pe = torch.empty((self.period, 192), dtype=torch.float32, device=dev)
            d = self.transformer_decoder.layers[0]
            dw = L.DecoderWeights()
            keep = {
                "sa_in_w": d.self_attn.in_proj_weight, "sa_in_b": d.self_attn.in_proj_bias,
                "sa_out_w": d.self_attn.out_proj.weight, "sa_out_b": d.self_attn.out_proj.bias,
                "ca_in_w": d.multihead_attn.in_proj_weight, "ca_in_b": d.multihead_attn.in_proj_bias,
                "ca_out_w": d.multihead_attn.out_proj.weight, "ca_out_b": d.multihead_attn.out_proj.bias,
                "lin1_w": d.linear1.weight, "lin1_b": d.linear1.bias, "lin2_w": d.linear2.weight, "lin2_b": d.linear2.bias,
                "n1_w": d.norm1.weight, "n1_b": d.norm1.bias, "n2_w": d.norm2.weight, "n2_b": d.norm2.bias,
                "n3_w": d.norm3.weight, "n3_b": d.norm3.bias, "fb_w": wc, "fb_b": bc,
                "obj_w": self.obj_vector.weight, "pe": self.PPE.pe, "fold_w": fold_w, "fold_pe": fold_pe,
            }
            for k_, v_ in keep.items():
                if not v_.is_contiguous():
                    raise L.A2FError(f"decoder parameter {k_} must be contiguous")
            keep = {k: v.detach() for k, v in keep.items()}         # the kernel reads the live parameters in place
            for k, v in keep.items():
                setattr(dw, k, v.data_ptr())
            P["dec"] = (dw, keep)
            plan.finalize()
            P["_plan"] = plan

            ca_mod = d.multihead_attn
            ca_srcs = (ca_mod.in_proj_weight, ca_mod.in_proj_bias, ca_mod.out_proj.weight, ca_mod.out_proj.bias,
                       self.audio_feature_map.weight, self.audio_feature_map.bias)
            fb_srcs = (self.vertice_map.weight, self.vertice_map.bias, self.vertice_map_r.weight, self.vertice_map_r.bias)

            def refresh(changed=None):
                # changed: data pointers of the sources modified since the last derivation (None = all)
                hit = lambda *ts: changed is None or any(t.data_ptr() in changed for t in ts)     # noqa: E731
                plan.run(changed)
                if hit(*ca_srcs):
                    fold_ca()
                if hit(pz.original0, pz.original1):
                    ops.pack_posconv_weight(pz.original0.detach().reshape(-1), pz.original1.detach(), dt, out=P["pos_w"])
                if hit(*fb_srcs):
                    ops.pack_feedback(self.vertice_map.weight.detach(), self.vertice_map.bias.detach(),
                                      self.vertice_map_r.weight.detach(), self.vertice_map_r.bias.detach(), out=(wc, bc))
                if hit(*fb_srcs, d.self_attn.in_proj_weight, self.PPE.pe):
                    ops.pack_decoder_fold(d.self_attn.in_proj_weight.detach(), wc, self.PPE.pe.detach(), self.period, fold_w,
                                          fold_pe)

            for p_ in (self.vertice_map.weight, self.vertice_map_r.weight, pz.original0, pz.original1):
                if not p_.is_contiguous():
                    raise L.A2FError("Faceformer parameters must be contiguous")
            P["_refresh"] = refresh
            refresh()
            return P

        srcs = list(self.parameters()) + [self.PPE.pe]
        return self._cache.get("ff_" + self.precision, srcs, build)

    # -- forward ----------------------------------------------------------------------------------------------
    def encode(self, audio: torch.Tensor, frame_num: int, stats: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Wav2Vec2Model.forward of ref:src/model/wav2vec.py:91-187 (processor normalisation included):
        raw audio [B,N] -> last_hidden_state [B*T,768] (bf16 or fp32 by precision).  `stats` [B,2] = (mean, rstd) of the
        processor's normalisation when the caller computes them differently (features.Wav2VecExtractor: one joint
        statistic for the whole batch); frame_num equal to the conv stack's output length makes the interpolation an
        identity, i.e. the plain HF Wav2Vec2Model."""
        P = self._packed()
        bf = self.precision == "bf16"
        dt = torch.bfloat16 if bf else torch.float32
        be = self._backend()
        ae = self.audio_encoder
        B, N = audio.shape
        dev = audio.device
        gn = ae.feature_extractor.conv_layers[0].layer_norm
        if stats is None:
            # processor statistics and conv0 moments from ONE pass over the raw audio (a2f_conv0_gn_gelu_auto)
            x, _ = ops.conv0_gn_gelu_auto(audio, P["conv0_w"], gn.weight.detach(), gn.bias.detach(), dt)
        else:
            x = ops.conv0_gn_gelu(audio, stats, P["conv0_w"], gn.weight.detach(), gn.bias.detach(), dt)   # [B,L0,512]
        L_in = x.shape[1]
        for i, k in enumerate((3, 3, 3, 3, 2, 2)):
            L_out = (L_in - k) // 2 + 1
            y = torch.empty((B, L_out, 512), dtype=dt, device=dev)
            ops.gemm(x, P["convs"][i], y, act=L.ACT_GELU, backend=be, M=B * L_out, K=k * 512, a_row_stride=1024,
                     a_batch_stride=L_in * 512, rows_per_batch=L_out, ldc=512)
            x, L_in = y, L_out
        T = frame_num
        fp = ae.feature_projection
        xi = ops.interp_ln(x, fp.layer_norm.weight.detach(), fp.layer_norm.bias.detach(), T, dt)       # [B,T,512]
        M = B * T
        h0 = torch.empty((M, 768), dtype=dt, device=dev)
        ops.gemm(xi.view(M, 512), P["proj_w"], h0, bias=fp.projection.bias.detach(), backend=be)
        pre = torch.empty((M, 768), dtype=dt, device=dev)
        ops.posconv(h0, P["pos_w"], ae.encoder.pos_conv_embed.conv.bias.detach(), pre, B, T, be)
        h = torch.empty((M, 768), dtype=dt, device=dev)
        ops.layernorm(pre, ae.encoder.layer_norm.weight.detach(), ae.encoder.layer_norm.bias.detach(), h)
        qkv = torch.empty((M, 2304), dtype=dt, device=dev)
        att = torch.empty((M, 768), dtype=dt, device=dev)
        ffn = torch.empty((M, 3072), dtype=dt, device=dev)
        layers = list(zip(ae.encoder.layers, P["layers"]))
        if bf:
            # everything of a layer but the attention is ONE kernel (a2f_encoder_block; cluster of three CTA pairs per 256-row
            # block): attention out-projection and its LayerNorm, W1, GELU, W2, residual, LayerNorm, and the NEXT layer's
            # q|k|v projection.  DESIGN.md section 4 has the timings.
            h1 = torch.empty((M, 768), dtype=dt, device=dev)
            h2 = torch.empty((M, 768), dtype=dt, device=dev)
            for i, (blk, W) in enumerate(layers):
                if i == 0:      # the later layers' q|k|v come out of the block kernel of the layer before
                    ops.gemm(h, W["qkv_w"], qkv, bias=W["qkv_b"], backend=be)
                ops.mha(qkv, att, B, T)
                kw = {}
                if i + 1 < len(layers):
                    nxt = layers[i + 1][1]
                    kw.update(wq=nxt["qkv_w"], bq=nxt["qkv_b"], qkv=qkv)
                ops.encoder_block(h1, W["f1_w"], blk.feed_forward.intermediate_dense.bias.detach(), W["f2_w"],
                                  blk.feed_forward.output_dense.bias.detach(), blk.final_layer_norm.weight.detach(),
                                  blk.final_layer_norm.bias.detach(), ffn, h2, att=att, wo=W["o_w"],
                                  bo=blk.attention.out_proj.bias.detach(), h_in=h, ln1_g=blk.layer_norm.weight.detach(),
                                  ln1_b=blk.layer_norm.bias.detach(), **kw)
                h, h2 = h2, h
            return h
        pre32 = torch.empty((M, 768), dtype=dt, device=dev)     # pre-LayerNorm sums
        for blk, W in layers:
            ops.gemm(h, W["qkv_w"], qkv, bias=W["qkv_b"], backend=be)
            ops.mha(qkv, att, B, T)
            ops.gemm(att, W["o_w"], pre32, bias=blk.attention.out_proj.bias.detach(), resid=h, backend=be)
            ops.layernorm(pre32, blk.layer_norm.weight.detach(), blk.layer_norm.bias.detach(), h)
            ops.gemm(h, W["f1_w"], ffn, bias=blk.feed_forward.intermediate_dense.bias.detach(), act=L.ACT_GELU, backend=be)
            ops.gemm(ffn, W["f2_w"], pre32, bias=blk.feed_forward.output_dense.bias.detach(), resid=h, backend=be)
            ops.layernorm(pre32, blk.final_layer_norm.weight.detach(), blk.final_layer_norm.bias.detach(), h)
        return h

    def forward(self, audio, one_hot, template, **kwargs):
        self._need_cuda(audio, one_hot, template)
        fps = int(kwargs.get("fps", self.fps))
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # training step: forward that keeps a tape + explicit backward kernels (training.py); gradients are
            # accumulated into every parameter's .grad by loss.backward()
            from . import training
            audio = audio.contiguous().float()
            if audio.dim() != 2:
                raise L.A2FError("audio must be [B, N] raw 16 kHz samples")
            B = audio.shape[0]
            if audio.shape[1] * fps // 16000 < 1:
                raise L.A2FError("audio too short for one output frame")
            return training.FaceformerTrainFn.run(self, audio, one_hot.reshape(B, -1).contiguous().float(),
                                                  template.reshape(B, -1).contiguous().float(), fps)
        audio = audio.contiguous().float()
        if audio.dim() != 2:
            raise L.A2FError("audio must be [B, N] raw 16 kHz samples")
        B, N = audio.shape
        frame_num = N * fps // 16000                                   # ref:faceformer.py:141
        if frame_num < 1:
            raise L.A2FError("audio too short for one output frame")
        one_hot = one_hot.reshape(B, -1).contiguous().float()
        tmpl = template.reshape(B, -1).contiguous().float()            # ref:faceformer.py:147
        # utterances are independent: a batch holding more than `max_chunk_seconds` of audio is ENCODED in utterance
        # chunks (bounds the conv0 activation, 16.4 MB bf16 per second of audio, and keeps element offsets inside
        # int32); the latency-bound decoder rollout then runs once for the whole batch (one CTA / cluster per utterance)
        per = max(1, int(min(float(kwargs.get("max_chunk_seconds", 480.0)) * 16000.0 / N, float(B))))
        P = self._packed()
        M = B * frame_num
        memory = torch.empty((M, 64), dtype=torch.float32, device=audio.device)
        for b0 in range(0, B, per):
            b1 = min(B, b0 + per)
            h = self.encode(audio[b0:b1], frame_num)
            ops.gemm(h, P["ca_w"], memory[b0 * frame_num:b1 * frame_num], bias=P["ca_b"], backend=self._backend())
            del h
        out = torch.empty((M, self.vertice_dim), dtype=torch.float32, device=audio.device)
        if self.stream_head and self.precision == "bf16" and ops.head_stream_supported(B, frame_num, self.vertice_dim):
            # rollout (one SM per utterance, T dependent steps) and vertex head (all other SMs, following frame group by
            # frame group) run at the same time; same bits as the two launches below
            ops.rollout_and_head_stream(P["dec"][0], memory, one_hot, self.period, B, frame_num,
                                        self._head_operand(self.vertice_map_r.weight, 64), self.vertice_map_r.bias.detach(),
                                        tmpl, out)
            return out.view(B, frame_num, -1, 3)
        D = ops.decoder_rollout(P["dec"][0], memory, one_hot, self.period, B, frame_num, memory_is_ca=True)
        hp = max(1, (1 << 17) // frame_num)                            # utterances per vertex-head launch (int32 offsets)
        for b0 in range(0, B, hp):
            b1 = min(B, b0 + hp)
            self._vertex_head(D.view(M, 64)[b0 * frame_num:b1 * frame_num], self.vertice_map_r.weight, self.vertice_map_r.bias,
                              tmpl[b0:b1], frame_num, 64, out=out[b0 * frame_num:b1 * frame_num])
        return out.view(B, frame_num, -1, 3)                           # ref:faceformer.py:187-188

    def predict(self, audio, one_hot, template, **kwargs):
        return self(audio, one_hot, template, **kwargs)


# ----------------------------------------------------------------------------------------------------------------
class _VocaLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, gt, k_rec, k_vel):
        rows = pred.shape[0]
        v3 = pred.numel() // rows
        p = pred.detach().reshape(rows, v3).contiguous().float()
        g = gt.detach().reshape(rows, v3).contiguous().float()
        out3 = ops.voca_loss_fwd(p, g, rows, v3, k_rec, k_vel)
        ctx.save_for_backward(p, g)
        ctx.meta = (rows, v3, k_rec, k_vel, pred.shape)
        ctx.mark_non_differentiable(out3)
        return out3[0].clone(), out3

    @staticmethod
    def backward(ctx, gloss, _gout3):
        p, g = ctx.saved_tensors
        rows, v3, k_rec, k_vel, shape = ctx.meta
        dpred = torch.empty_like(p)
        ops.voca_loss_bwd(p, g, rows, v3, k_rec, k_vel, gloss.contiguous().float(), dpred)
        return dpred.view(shape), None, None, None


class VocaLoss:
    """Drop-in for ref:src/loss/loss.py:24-55: returns {"loss", "rec_loss", "vel_loss"} 0-d tensors, `loss`
    differentiable w.r.t. pred."""

    def __init__(self, k_rec: float = 1.0, k_vel: float = 10.0):
        self.k_rec = k_rec
        self.k_vel = k_vel

    def __call__(self, pred, gt):
        if not pred.is_cuda:
            raise L.A2FError("VocaLoss runs on CUDA (sm_100a) only")
        bs = pred.shape[0]
        if bs % 2 != 0:
            raise L.A2FError("VocaLoss needs an even number of rows (ref loss.py:34 views pairs of consecutive frames)")
        self.n_verts = pred.numel() // bs // 3
        loss, out3 = _VocaLossFn.apply(pred, gt, float(self.k_rec), float(self.k_vel))
        return {"loss": loss, "rec_loss": out3[1], "vel_loss": out3[2]}


class FaceFormerLoss:
    """Drop-in for ref:src/loss/loss.py:4-17."""

    def __init__(self) -> None:
        self.loss = VocaLoss()

    def __call__(self, pred, gt):
        if pred.dim() == 4 and pred.shape[0] > 1:
            # batch extension (the reference is batch-1, SURVEY.md fact 0.4): mean of the per-utterance losses.  With an
            # even number of frames per utterance the velocity pairs (2k, 2k+1) never straddle two utterances, so this
            # is VocaLoss over the [B*T, V3] rows.
            if gt.shape[1] % 2 != 0:
                gt = gt[:, :-1]
                pred = pred[:, :-1]
            return self.loss(pred.reshape(-1, pred.shape[2], pred.shape[3]), gt.reshape(-1, gt.shape[2], gt.shape[3]))
        gt = gt.squeeze(0)
        pred = pred.squeeze(0)
        if gt.shape[0] % 2 != 0:      # drop the last frame of an odd-length clip
            gt = gt[:-1]
            pred = pred[:-1]
        return self.loss(pred, gt)


def mse_error(pred: torch.Tensor, gt: torch.Tensor) -> torch.Tensor:
    """ref:src/model/lightning_model.py:119-125: mean_b mean_15069 (p-g)^2 == rec_loss / 3 (one fused pass)."""
    rows = pred.numel() // (5023 * 3)
    if rows < 1 or not pred.is_cuda:
        raise L.A2FError("mse_error runs on CUDA (sm_100a) only and needs at least one frame")
    p = pred.detach().reshape(rows, -1).contiguous().float()
    g = gt.detach().reshape(rows, -1).contiguous().float()
    v3 = p.shape[1]
    even = rows - (rows % 2)
    acc = None
    if even:
        acc = ops.voca_loss_fwd(p, g, even, v3, 1.0, 0.0)[1] * (even / rows)
    if rows % 2:
        # any frame count is legal here (the reference calls mse_error on the FULL prediction, odd-length FaceFormer
        # clips included, ref:lightning_model.py:119-125,156): the paired-row kernel takes the last row twice
        lp, lg = p[rows - 1:].expand(2, v3).contiguous(), g[rows - 1:].expand(2, v3).contiguous()
        last = ops.voca_loss_fwd(lp, lg, 2, v3, 1.0, 0.0)[1] * (1.0 / rows)
        acc = last if acc is None else acc + last
    return acc / 3.0
